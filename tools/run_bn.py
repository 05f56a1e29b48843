"""Time the fused BN + residual + PReLU kernels (forward and backward) at the model's two layout cases.
    python tools/run_bn.py [--n 256] [--sync]

--sync also times the synchronised BatchNorm phases (dstd_bn_act_{forward,backward}_{local,global}) and the fp64
row exchange between them (a one-rank all_gather over NCCL: the collective's fixed cost, no inter-GPU traffic).
"""
import argparse
import os
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from dstd_gcn_b200 import _lib          # noqa: E402
from dstd_gcn_b200.ops import _out_like  # noqa: E402


def _graph_us(fn, reps):
    """Device time of fn per call, replayed as a CUDA graph (no host gaps)."""
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    g.replay()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    e[0].record()
    for _ in range(reps):
        g.replay()
    e[1].record()
    torch.cuda.synchronize()
    return e[0].elapsed_time(e[1]) * 1e3 / reps


def _eager_us(fn, reps):
    """Wall time per call on the stream, host launch cost included."""
    fn()
    torch.cuda.synchronize()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    e[0].record()
    for _ in range(reps):
        fn()
    e[1].record()
    torch.cuda.synchronize()
    return e[0].elapsed_time(e[1]) * 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--gr-add", action="store_true", help="backward with a gr_add tensor (layer-skip gradient)")
    ap.add_argument("--sync", action="store_true", help="also time the synchronised-BN phases and the exchange")
    a = ap.parse_args()
    dev, be = torch.device("cuda"), _lib.backend()
    n, c, t, v = a.n, 64, 35, 22
    g = torch.Generator().manual_seed(0)
    gamma, beta = torch.ones(c * v, device=dev), torch.zeros(c * v, device=dev)
    rm, rv, nbt = torch.zeros(c * v, device=dev), torch.ones(c * v, device=dev), torch.zeros((), dtype=torch.int64, device=dev)
    prelu = torch.tensor([0.25], device=dev)
    cases = {
        "block BN  (y T-major, r T-major -> out V-major)": (torch.randn(n, c, t, v, generator=g).to(dev),
                                                            torch.randn(n, c, t, v, generator=g).to(dev), 2),
        "encoder BN (y V-major -> out T-major)": (torch.randn(n, c, v, t, generator=g).to(dev).permute(0, 1, 3, 2), None, 1),
    }
    tmp = tempfile.TemporaryDirectory() if a.sync else None     # the one-rank group's FileStore; removed at exit
    if a.sync:
        import torch.distributed as dist
        dist.init_process_group("nccl", store=dist.FileStore(os.path.join(tmp.name, "store"), 1), rank=0, world_size=1,
                                device_id=torch.device("cuda", torch.cuda.current_device()))
    try:
        for name, (y, r, order) in cases.items():
            ol = _out_like(y, order)
            out, mean, istd = be.bn_act_forward(y, r, gamma, beta, rm, rv, nbt, prelu, None, False, True, 1e-5, 0.1, ol)
            gout = out    # any tensor with the output's layout
            gadd = torch.randn_like(gout) if (a.gr_add and r is not None) else None
            fwd = lambda: be.bn_act_forward(y, r, gamma, beta, rm, rv, nbt, prelu, None, False, True, 1e-5, 0.1, ol)
            bwd = lambda: be.bn_act_backward(y, r, gout, gamma, beta, prelu, None, mean, istd, False, True, True, gadd)
            pf, pb = _graph_us(fwd, a.reps), _graph_us(bwd, a.reps)
            print(f"{name}: fwd {pf:.1f} us  bwd {pb:.1f} us")
            if not a.sync:
                continue
            rows = be.bn_act_forward_local(y, False)
            _, _, _, brows, gy, gr = be.bn_act_backward_local(y, r, gout, gamma, beta, prelu, None, mean, istd, False,
                                                              True, gadd)
            parts = [torch.empty_like(rows)]
            f_loc = lambda: be.bn_act_forward_local(y, False)
            f_glo = lambda: be.bn_act_forward_global(y, r, gamma, beta, rm, rv, nbt, prelu, None, False, 1e-5, 0.1,
                                                     rows, ol)
            b_loc = lambda: be.bn_act_backward_local(y, r, gout, gamma, beta, prelu, None, mean, istd, False, True, gadd)
            b_glo = lambda: be.bn_act_backward_global(y, r, gout, gamma, beta, prelu, None, mean, istd, False, brows,
                                                      gy, gr, gadd)

            def gather():
                dist.all_gather(parts, rows)
                return torch.cat(parts)

            def f_split():
                rr = be.bn_act_forward_local(y, False)
                dist.all_gather(parts, rr)
                be.bn_act_forward_global(y, r, gamma, beta, rm, rv, nbt, prelu, None, False, 1e-5, 0.1,
                                         torch.cat(parts), ol)

            def b_split():
                res = be.bn_act_backward_local(y, r, gout, gamma, beta, prelu, None, mean, istd, False, True, gadd)
                dist.all_gather(parts, res[3])
                be.bn_act_backward_global(y, r, gout, gamma, beta, prelu, None, mean, istd, False, torch.cat(parts),
                                          res[4], res[5], gadd)

            print(f"  sync phases (graph): fwd local {_graph_us(f_loc, a.reps):.1f} + global {_graph_us(f_glo, a.reps):.1f} us"
                  f"   bwd local {_graph_us(b_loc, a.reps):.1f} + global {_graph_us(b_glo, a.reps):.1f} us")
            print(f"  one-rank all_gather of {rows.numel() * 8 / 1000:.1f} kB fp64 + cat (eager): "
                  f"{_eager_us(gather, a.reps):.1f} us")
            print(f"  eager end to end: fwd plain {_eager_us(fwd, a.reps):.1f} / split {_eager_us(f_split, a.reps):.1f} us"
                  f"   bwd plain {_eager_us(bwd, a.reps):.1f} / split {_eager_us(b_split, a.reps):.1f} us")
    finally:
        if a.sync:
            dist.destroy_process_group()
            tmp.cleanup()


if __name__ == "__main__":
    main()
