"""Synchronised BatchNorm (``ops.sync_batch_norm``, ``TrainStep(sync_bn=True)``): each training-mode BN call runs a
local phase, an all-gather of fp64 rows in rank order and a global phase, and must compute what one plain BN call on
the concatenated batch computes.

CPU: the four ABI phases in the fp64 emulation against the emulated plain call; two gloo ranks running
``TrainStep(sync_bn=True)`` against the oracle's single-process step on the full batch; the ctypes prototypes.
GPU: the four entry points against the plain ones on the concatenated batch; two processes over gloo on one GPU and
two ranks over NCCL on two GPUs against the single-process step on the full batch; one process unchanged."""
import ctypes
import os
import re
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests.helpers import load_npz, max_abs, split

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "dstd_b200.h")
SYNC_SYMBOLS = ("dstd_bn_sync_buffer_doubles", "dstd_bn_act_forward_local", "dstd_bn_act_forward_global",
                "dstd_bn_act_backward_local", "dstd_bn_act_backward_global")


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _ordered(g, n, c, t, v, order, dtype=torch.float64):
    if order == "t":
        return torch.randn((n, c, t, v), generator=g, dtype=dtype)
    return torch.randn((n, c, v, t), generator=g, dtype=dtype).permute(0, 1, 3, 2)


def _shard(x, lo, hi):
    """A rank's own copy of samples lo..hi, in x's memory order."""
    if x is None:
        return None
    s = x[lo:hi]
    return torch.empty_like(s).copy_(s)


def _bounds(sizes):
    b = [0]
    for s in sizes:
        b.append(b[-1] + s)
    return list(zip(b[:-1], b[1:]))


def _sync_bn_vs_plain(be, n_shards, c, t, v, yo, ro, vc, use_prelu, use_mask, dev, dtype, gen_seed, check_twice=False):
    """Runs sharded local -> concatenate -> global through backend `be` and the plain call on the whole batch.
    Returns (plain results, sync results) as dicts of comparable tensors."""
    from dstd_gcn_b200.ops import _out_like
    g = torch.Generator().manual_seed(gen_seed)
    n = sum(n_shards)
    to = (lambda x: None if x is None else x.to(dev, dtype))
    y = to(_ordered(g, n, c, t, v, yo) * 2.0 + 3.0)
    r = to(_ordered(g, n, c, t, v, ro)) if ro else None
    gamma, beta = to(torch.randn(c * v, generator=g, dtype=torch.float64) * 0.5 + 1.0), \
        to(torch.randn(c * v, generator=g, dtype=torch.float64) * 0.5)
    rm0, rv0 = to(torch.randn(c * v, generator=g, dtype=torch.float64) * 0.5), \
        to(torch.rand(c * v, generator=g, dtype=torch.float64) + 0.5)
    prelu = to(torch.tensor([0.25], dtype=torch.float64)) if use_prelu else None
    mask = to((torch.rand((n, c, t, v), generator=g) > 0.1).double() / 0.9) if use_mask else None
    out_order = 2 if yo == "t" else 1
    ol = _out_like(y, out_order)
    gout = torch.empty_like(ol, device=dev).copy_(to(torch.randn(tuple(y.shape), generator=g, dtype=torch.float64)))
    gadd = torch.empty_like(gout).copy_(to(torch.randn(tuple(y.shape), generator=g, dtype=torch.float64))) if r is not None else None
    eps, mom = 1e-5, 0.1

    # plain call on the whole batch
    rm, rv, nbt = rm0.clone(), rv0.clone(), torch.tensor(3, dtype=torch.int64, device=dev)
    out, mean, istd = be.bn_act_forward(y, r, gamma, beta, rm, rv, nbt, prelu, mask, vc, True, eps, mom, ol)
    gy, gr, gg, gb, gp = be.bn_act_backward(y, r, gout, gamma, beta, prelu, mask, mean, istd, vc, True, True, gadd)
    plain = dict(out=out, mean=mean, istd=istd, rm=rm, rv=rv, nbt=nbt, gy=gy, gr=gr, gg=gg, gb=gb, gp=gp)

    # the shards: local phases, "all-gather" (concatenation in rank order), global phases
    sh = [dict(y=_shard(y, lo, hi), r=_shard(r, lo, hi), mask=_shard(mask, lo, hi), gout=_shard(gout, lo, hi),
               gadd=_shard(gadd, lo, hi)) for lo, hi in _bounds(n_shards)]
    rows = torch.cat([be.bn_act_forward_local(s["y"], vc) for s in sh])
    fwd = []
    for s in sh:
        rm_k, rv_k, nbt_k = rm0.clone(), rv0.clone(), torch.tensor(3, dtype=torch.int64, device=dev)
        o, m, i = be.bn_act_forward_global(s["y"], s["r"], gamma, beta, rm_k, rv_k, nbt_k, prelu, s["mask"], vc, eps,
                                           mom, rows, _out_like(s["y"], out_order))
        fwd.append((o, m, i, rm_k, rv_k, nbt_k))
    loc = [be.bn_act_backward_local(s["y"], s["r"], s["gout"], gamma, beta, prelu, s["mask"], fwd[k][1], fwd[k][2],
                                    vc, True, s["gadd"]) for k, s in enumerate(sh)]
    brows = torch.cat([l_[3] for l_ in loc])
    bwd = [be.bn_act_backward_global(s["y"], s["r"], s["gout"], gamma, beta, prelu, s["mask"], fwd[k][1], fwd[k][2],
                                     vc, brows, loc[k][4], loc[k][5], s["gadd"]) for k, s in enumerate(sh)]
    # replicas: identical gathered rows give identical statistics and running statistics on every rank
    for f in fwd[1:]:
        for a, b in zip(f[1:], fwd[0][1:]):
            assert torch.equal(a, b)
    if check_twice:
        s, f = sh[0], fwd[0]
        rm_k, rv_k, nbt_k = rm0.clone(), rv0.clone(), torch.tensor(3, dtype=torch.int64, device=dev)
        again = be.bn_act_forward_global(s["y"], s["r"], gamma, beta, rm_k, rv_k, nbt_k, prelu, s["mask"], vc, eps,
                                         mom, rows, _out_like(s["y"], out_order))
        for a, b in zip(again + (rm_k, rv_k, nbt_k), f):
            assert torch.equal(a, b)
        gy2 = torch.empty_like(loc[0][4])
        gr2 = torch.empty_like(loc[0][5]) if loc[0][5] is not None else None
        again = be.bn_act_backward_global(s["y"], s["r"], s["gout"], gamma, beta, prelu, s["mask"], f[1], f[2], vc,
                                          brows, gy2, gr2, s["gadd"])
        for a, b in zip(again, bwd[0]):
            assert (a is None and b is None) or torch.equal(a, b)
    for f in fwd:     # each rank's output in the layout the plain call gives (the concatenation below is contiguous)
        assert f[0].stride() == out.stride()
    sync = dict(out=torch.cat([f[0] for f in fwd]), mean=fwd[0][1], istd=fwd[0][2], rm=fwd[0][3], rv=fwd[0][4],
                nbt=fwd[0][5], gy=torch.cat([b[0] for b in bwd]),
                gr=torch.cat([b[1] for b in bwd]) if r is not None else None,
                gg=sum(l_[0] for l_ in loc), gb=sum(l_[1] for l_ in loc),
                gp=sum(l_[2] for l_ in loc) if use_prelu else None)
    return plain, sync


# ====================================================================================================== CPU
EMUL_CASES = [
    # vc_order, residual, prelu, mask
    (False, True, True, False),
    (True, False, False, False),
    (False, False, True, True),
    (True, True, True, True),
]


@pytest.mark.parametrize("case", EMUL_CASES, ids=["res_prelu", "vc_plain", "prelu_mask", "vc_res_prelu_mask"])
def test_emulated_abi_phases_equal_plain_call_on_whole_batch(case):
    from tests.bn_sync_emul import SyncEmulBackend
    vc, use_r, use_prelu, use_mask = case
    be = SyncEmulBackend()
    plain, sync = _sync_bn_vs_plain(be, [3, 5], 4, 7, 5, "t" if use_r else "v", "t" if use_r else None, vc,
                                    use_prelu, use_mask, "cpu", torch.float64, 11)
    for k, ref in plain.items():
        if ref is None:
            assert sync[k] is None, k
            continue
        assert sync[k].shape == ref.shape, k
        assert max_abs(sync[k], ref) <= 1e-12 * max(1.0, float(ref.double().abs().max())), k


def _gloo_worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.set_num_threads(1)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import dstd_gcn_b200  # noqa: F401
        from dstd_gcn_b200 import _lib, ops
        from dstd_gcn_b200.engine import TrainStep
        from dstd_gcn_b200.model import dstdgcn as std
        from tests.bn_sync_emul import SyncEmulBackend
        _lib._set_backend_for_tests(SyncEmulBackend())
        z = load_npz("train_std.npz")
        m = std.DSTDGCN(6, 4, 6, 0.0, 22, 8, 2, "h36m").double()
        m.load_state_dict({k: v.clone() for k, v in split(z, "p.").items()})
        m.train()
        step = TrainStep(m, lr=3e-3, inverse=True, sync_bn=True)
        assert step.sync_bn
        for s in range(2):
            sl = slice(rank * 2, rank * 2 + 2)
            step(z[f"inputs{s}"][sl].contiguous(), z[f"inputs_inv{s}"][sl].contiguous(),
                 z[f"targets{s}"][sl].contiguous())
        errors = []
        try:
            step.capture(z["inputs0"][:2], z["inputs_inv0"][:2], z["targets0"][:2])
        except RuntimeError as e:
            errors.append("capture" if "eagerly" in str(e) else repr(e))
        try:
            with ops.sync_batch_norm(), ops.defer_bn_updates():
                pass
        except RuntimeError as e:
            errors.append("defer" if "defer_bn_updates" in str(e) else repr(e))
        sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
        bufs = torch.cat([b.double().reshape(-1) for _, b in m.named_buffers()])
        gathered = [torch.zeros_like(bufs) for _ in range(world)]
        dist.all_gather(gathered, bufs)
        if rank == 0:
            q.put(("ok", errors, [g.numpy() for g in gathered], {k: v.numpy() for k, v in sd.items()}))
    except Exception as e:  # pragma: no cover
        if rank == 0:
            q.put(("err", repr(e), None, None))
        raise
    finally:
        dist.destroy_process_group()


def _oracle_full_batch(steps):
    """The oracle's single-process step on the whole 4-sample batch, torch Adam."""
    from oracle import dstd_oracle as orc
    from dstd_gcn_b200.model import dstdgcn as std
    z = load_npz("train_std.npz")
    p = {k: v.clone() for k, v in split(z, "p.").items()}
    m = std.DSTDGCN(6, 4, 6, 0.0, 22, 8, 2, "h36m").double()
    req = {k: prm.requires_grad for k, prm in m.named_parameters()}
    params = {k: v.requires_grad_(True) for k, v in p.items() if req.get(k, False)}
    opt = torch.optim.Adam(list(params.values()), lr=3e-3)
    for s in range(steps):
        loss = orc.train_loss(p, z[f"inputs{s}"], z[f"inputs_inv{s}"], z[f"targets{s}"])
        gs = torch.autograd.grad(loss, list(params.values()), allow_unused=True)
        for (k, v), g in zip(params.items(), gs):
            v.grad = g if g is not None else torch.zeros_like(v)
        opt.step()
    return {k: v.detach() for k, v in p.items()}


@pytest.mark.timeout(600)
def test_two_gloo_ranks_with_sync_bn_match_single_process_full_batch():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, world, port, q)) for r in range(world)]
    try:
        for pr in procs:
            pr.start()
        status, errors, bufs, sd = q.get(timeout=500)
        for pr in procs:
            pr.join(timeout=120)
            assert pr.exitcode == 0
    finally:
        for pr in procs:
            if pr.is_alive():
                pr.terminate()
                pr.join()
    assert status == "ok", errors
    assert errors == ["capture", "defer"]
    assert np.array_equal(bufs[0], bufs[1])             # running statistics bit-identical across the ranks
    ref = _oracle_full_batch(2)
    for k, v in ref.items():
        if k.endswith("residual.0.bias") or not v.is_floating_point():
            continue                            # zero true gradient: Adam turns rounding noise into +-lr steps
        got = torch.from_numpy(sd[k])
        assert float((got - v).abs().max()) <= 1e-10 * max(1.0, float(v.abs().max())), k


def _header_prototype(name):
    src = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    m = re.search(r"([A-Za-z_][\w\s\*]*?)\b" + name + r"\s*\(([^)]*)\)\s*;", src)
    ret = m.group(1).split()[-1] if "*" not in m.group(1) else "ptr"
    args = []
    for a in m.group(2).split(","):
        a = a.strip()
        if "*" in a:
            args.append("args*" if "_args" in a else "ptr")
        else:
            args.append(a.rsplit(None, 1)[0].replace("const ", ""))
    return ret, args


_CTYPE = {"int": ctypes.c_int, "size_t": ctypes.c_size_t, "dstd_stream_t": ctypes.c_void_p, "ptr": ctypes.c_void_p}


def test_sync_symbols_ctypes_prototypes_match_header():
    import __graft_entry__ as entry
    from dstd_gcn_b200 import _lib
    entry.build()
    lib = _lib.load_library()
    for name in SYNC_SYMBOLS:
        assert hasattr(lib, name), name
        ret, args = _header_prototype(name)
        res, argtypes = _lib.SYMBOLS[name]
        assert res is _CTYPE[ret], name
        assert len(argtypes) == len(args), name
        for a, t in zip(args, argtypes):
            if a == "args*":
                assert issubclass(t, ctypes._Pointer) and t._type_ in (_lib.BnFwdArgs, _lib.BnBwdArgs), name
            else:
                assert t is _CTYPE[a], (name, a)
    assert lib.dstd_bn_sync_buffer_doubles(64, 22) == 3 * 64 * 22
    # training = 0 is refused before anything touches a device
    a = _lib.BnFwdArgs()
    a.training = 0
    assert lib.dstd_bn_act_forward_local(ctypes.byref(a), None, None) == -1
    assert b"training" in lib.dstd_last_error()
    b = _lib.BnBwdArgs()
    b.training = 0
    assert lib.dstd_bn_act_backward_global(ctypes.byref(b), None, 1, None) == -1


# ====================================================================================================== GPU
DEV = "cuda"

GPU_CASES = {
    # name: (shard sizes, c, t, v, y_order, r_order, vc_order, prelu, mask)
    "block_res": ([2, 2], 16, 35, 22, "t", "t", False, True, False),
    "encoder_mask": ([2, 2], 16, 35, 22, "v", None, False, True, True),
    "vc_plain": ([1, 2], 8, 10, 25, "t", None, True, False, False),
    "many_splits": ([24, 16], 64, 35, 22, "v", None, False, True, False),
    "out_block": ([1, 1], 3, 35, 22, "t", "t", False, True, False),
    "h36m_block_fast": ([37, 27], 64, 35, 22, "t", "t", False, True, False),
    "stress_slab_big": ([3, 2], 4, 125, 22, "t", "t", False, True, False),
    "stress_layer": ([2, 1], 4, 125, 22, "v", None, False, True, False),
    "unequal_three": ([1, 6, 2], 8, 35, 22, "t", "t", False, True, False),
}


@pytest.mark.gpu
@pytest.mark.parametrize("fast", ["1", "0"])
@pytest.mark.parametrize("name", list(GPU_CASES))
def test_sync_abi_on_device_equals_plain_call(name, fast, monkeypatch):
    from dstd_gcn_b200 import _lib
    monkeypatch.setenv("DSTD_BN_FAST", fast)
    shards, c, t, v, yo, ro, vc, use_prelu, use_mask = GPU_CASES[name]
    be = _lib.CudaBackend()
    plain, sync = _sync_bn_vs_plain(be, shards, c, t, v, yo, ro, vc, use_prelu, use_mask, DEV, torch.float32,
                                    sum(shards) * 31 + c, check_twice=True)
    torch.cuda.synchronize()
    assert be.lib.dstd_device_error(0) == 0
    for k in ("out", "mean", "istd", "rm", "rv"):
        ref = plain[k].double().cpu()
        assert max_abs(sync[k], ref) <= 1e-5 * max(1.0, float(ref.abs().max())), k
    assert int(sync["nbt"]) == int(plain["nbt"]) == 4
    for k in ("gy", "gr", "gg", "gb", "gp"):
        ref = plain[k]
        if ref is None:
            assert sync[k] is None, k
            continue
        ref = ref.double().cpu()
        assert max_abs(sync[k], ref) <= 1e-4 * max(1.0, float(ref.abs().max())), k


def _gpu_model():
    from dstd_gcn_b200.model import dstdgcn as std
    torch.manual_seed(777)
    return std.DSTDGCN(6, 10, 25, 0.0, 22, 16, 2, "h36m")


def _gpu_batch(n):
    g = torch.Generator().manual_seed(3)
    inputs = torch.randn(n, 35, 66, generator=g)
    return inputs, torch.flip(inputs, dims=[1]).contiguous(), inputs + 0.1 * torch.randn(n, 35, 66, generator=g)


def _dp_worker(rank, world, port, backend, shard, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = torch.device("cuda", rank if backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    dist.init_process_group(backend, rank=rank, world_size=world)
    try:
        from dstd_gcn_b200.engine import TrainStep
        m = _gpu_model().to(dev).train()
        step = TrainStep(m, lr=3e-3, inverse=True, sync_bn=True)
        assert step.sync_bn
        inputs, inputs_inv, targets = (x[rank * shard:(rank + 1) * shard].to(dev) for x in _gpu_batch(world * shard))
        loss = step(inputs, inputs_inv, targets)
        # numpy, not tensors: the queue would share tensors through file descriptors of a process about to exit
        first = (float(loss), (step.flat.grad.double().cpu() / world).numpy(),
                 {k: b.double().cpu().numpy() for k, b in m.named_buffers()})
        for _ in range(2):
            step(inputs, inputs_inv, targets)
        state = torch.cat([step.flat.param.double()] + [b.double().reshape(-1) for _, b in m.named_buffers()])
        gathered = [torch.zeros_like(state) for _ in range(world)]
        dist.all_gather(gathered, state)
        torch.cuda.synchronize()
        if rank == 0:
            q.put(("ok", first, [x.cpu().numpy() for x in gathered]))
        else:
            q.put(("loss", float(first[0]), None))
    except Exception as e:  # pragma: no cover
        q.put(("err", repr(e), None))
        raise
    finally:
        dist.destroy_process_group()


def _run_dp(backend, world, shard):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, backend, shard, q)) for r in range(world)]
    try:
        for pr in procs:
            pr.start()
        msgs = [q.get(timeout=600) for _ in range(world)]
        for pr in procs:
            pr.join(timeout=120)
            assert pr.exitcode == 0
    finally:
        for pr in procs:
            if pr.is_alive():
                pr.terminate()
                pr.join()
    errs = [m for m in msgs if m[0] == "err"]
    assert not errs, errs
    ok = next(m for m in msgs if m[0] == "ok")
    other_losses = [m[1] for m in msgs if m[0] == "loss"]
    return ok[1], ok[2], other_losses


def _check_dp_against_full_batch(backend, world, shard):
    from dstd_gcn_b200.engine import TrainStep
    (loss0, grad, bufs), states, other_losses = _run_dp(backend, world, shard)
    # the plain single-process step on the whole batch
    m = _gpu_model().to(DEV).train()
    step = TrainStep(m, lr=3e-3, inverse=True)
    full = step(*(x.to(DEV) for x in _gpu_batch(world * shard)))
    torch.cuda.synchronize()
    mean_loss = (loss0 + sum(other_losses)) / world
    assert abs(mean_loss - float(full)) <= 1e-5 * max(1.0, abs(float(full)))
    gref = step.flat.grad.double().cpu()
    assert float((torch.from_numpy(grad) - gref).abs().max()) <= 1e-4 * float(gref.abs().max())
    for k, b in m.named_buffers():
        got = torch.from_numpy(bufs[k])
        if not b.is_floating_point():
            assert int(got) == int(b), k
            continue
        ref = b.double().cpu()
        assert max_abs(got, ref) <= 1e-5 * max(1.0, float(ref.abs().max())), k
    for s in states[1:]:
        assert np.array_equal(s, states[0])        # replicas bit-identical after 3 steps


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_two_processes_on_one_gpu_over_gloo_match_full_batch():
    _check_dp_against_full_batch("gloo", 2, 8)


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_two_ranks_over_nccl_match_full_batch():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _check_dp_against_full_batch("nccl", 2, 8)


@pytest.mark.gpu
@pytest.mark.parametrize("captured", [False, True], ids=["eager", "captured"])
def test_sync_bn_single_process_is_the_default_path(captured):
    from dstd_gcn_b200.engine import TrainStep
    batch = tuple(x.to(DEV) for x in _gpu_batch(8))
    res = []
    for sync in (False, True):
        m = _gpu_model().to(DEV).train()
        step = TrainStep(m, lr=3e-3, inverse=True, sync_bn=sync)
        assert not step.sync_bn
        if captured:
            step.capture(*batch)
        losses = [step(*batch).clone() for _ in range(2)]
        torch.cuda.synchronize()
        res.append((losses, step.flat.param.clone(), [b.clone() for b in m.buffers()]))
    (la, pa, ba), (lb, pb, bb) = res
    assert all(torch.equal(x, y) for x, y in zip(la, lb))
    assert torch.equal(pa, pb)
    assert all(torch.equal(x, y) for x, y in zip(ba, bb))
