"""Pose sequences of any coordinate count D (1 <= D <= 32): DSTDGCN(input_channels = 2 * D) on x [N, T, V, D], as the
reference's ``input_channels`` allows (model/dstdgcn.py:298-303: cat(x, x - x_last) has 2D channels, conv_st_out returns
input_channels // 2).

CPU: an fp64 restatement of the reference head, tail and loss for any D (equal to the oracle's at D = 3), the ABI
emulation for D against autograd of it, a D = 2 model through the host wiring, the input validation, ``mirror``,
``window_batch`` and ``evaluate`` at D = 2, and the new ctypes prototypes against the header.
GPU: every new entry point against the emulation at D = 1, 2, 4, 32, the D = 3 bits of the original entry points,
whole models and training steps at D = 2 and 4, and the kernels a training step launches."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from dstd_gcn_b200 import _lib, data, engine
from oracle import dstd_oracle as orc
from oracle.abi_emul import EmulBackend
from tests.helpers import max_abs, rel_err
from tests.pose_dims_emul import PoseDimsEmulBackend

DEV = "cuda"
EM = PoseDimsEmulBackend()
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ====================================================================================== restatement of the reference
def head(x):
    """DSTDGCN.forward's input (model/dstdgcn.py:298-303): [N,T,V,D] -> [N,T,V,2D]."""
    return torch.cat((x, x - x[:, -1:]), dim=-1)


def tail(z, x):
    """The last observed frame added back (model/dstdgcn.py:314-315): z [N,T,V,D]."""
    return z + x[:, -1:]


def pose_loss(outputs, targets, d):
    """mpjpe_error_3d (engine/utils/loss.py:52-65) over D-vectors."""
    diff = outputs.reshape(-1, d) - targets.reshape(-1, d)
    return torch.sqrt((diff * diff).sum(dim=1)).mean()


def train_loss(p, inputs, inputs_inv, targets, d, fast=False, dropout_masks=(None, None)):
    """orc.train_loss (engine/prediction.py:223-287) on [N,T,D*V] batches."""
    n, t, vc = inputs.shape
    out = orc.dstdgcn(inputs.view(n, t, vc // d, d), p, True, fast, dropout_masks[0]).reshape(n, t, vc)
    out_i = orc.dstdgcn(inputs_inv.view(n, t, vc // d, d), p, True, fast, dropout_masks[1]).reshape(n, t, vc)
    return (pose_loss(out, targets, d) + pose_loss(out_i, torch.flip(targets, dims=[1]), d)) / 2


def _mod(variant):
    from dstd_gcn_b200.model import dstdgcn, dstdgcn_fast
    return dstdgcn if variant == "std" else dstdgcn_fast


def _perturbed(m):
    with torch.no_grad():
        for k, p in m.named_parameters():
            leaf = k.split(".")[-1]
            if leaf in ("alpha_sm", "alpha_tm"):
                p.fill_(0.1)
            elif leaf == "W_s":
                p.fill_(0.05)
            elif leaf == "R_t":
                p.fill_(0.01)
    return m


# ====================================================================================================== CPU
def test_restatement_equals_oracle_at_xyz():
    g = torch.Generator().manual_seed(1)
    x = torch.randn(3, 8, 22, 3, generator=g, dtype=torch.float64)
    out, tgt = torch.randn(3, 8, 66, generator=g, dtype=torch.float64), torch.randn(3, 8, 66, generator=g,
                                                                                      dtype=torch.float64)
    assert torch.equal(pose_loss(out, tgt, 3), orc.mpjpe(out, tgt))
    torch.manual_seed(777)
    m = _perturbed(_mod("std").DSTDGCN(6, 3, 5, 0.0, 22, 8, 1, "h36m"))
    p = orc.state_from_module(m, torch.float64)
    a, b = torch.randn(2, 8, 66, generator=g, dtype=torch.float64), torch.randn(2, 8, 66, generator=g,
                                                                                dtype=torch.float64)
    assert torch.equal(train_loss(p, a, b, tgt[:2], 3), orc.train_loss(p, a, b, tgt[:2]))
    # the oracle's ABI emulation of the xyz head and tail
    xyz = EmulBackend()
    z = torch.randn(3, 3, 8, 22, generator=g, dtype=torch.float64)
    assert torch.equal(xyz.prep_forward(x), head(x).permute(0, 3, 1, 2))
    assert torch.equal(xyz.finish_forward(z, x), tail(z.permute(0, 2, 3, 1), x))
    l_xyz, l_d = torch.zeros((), dtype=torch.float64), torch.zeros((), dtype=torch.float64)
    assert torch.equal(xyz.mpjpe(out, tgt, 0.5, l_xyz, False), EM.pose_error(out, tgt, 0.5, l_d, False, 3))
    assert torch.equal(l_xyz, l_d) and torch.equal(l_d, 0.5 * pose_loss(out, tgt, 3))
    gh = torch.randn(3, 6, 8, 22, generator=g, dtype=torch.float64)
    assert torch.equal(xyz.prep_backward(gh), EM.prep_backward(gh))


@pytest.mark.parametrize("d", [1, 2, 4])
def test_emulation_vs_autograd_of_restatement(d):
    g = torch.Generator().manual_seed(10 + d)
    n, t, v = 3, 7, 5
    x = torch.randn(n, t, v, d, generator=g, dtype=torch.float64, requires_grad=True)
    h = head(x).permute(0, 3, 1, 2)
    assert torch.equal(EM.prep_forward(x.detach()), h.detach())
    gh = torch.randn(n, 2 * d, t, v, generator=g, dtype=torch.float64)
    (gx,) = torch.autograd.grad(h, x, gh)
    assert max_abs(EM.prep_backward(gh), gx) < 1e-13
    z = torch.randn(n, d, t, v, generator=g, dtype=torch.float64, requires_grad=True)
    y = tail(z.permute(0, 2, 3, 1), x)
    assert torch.equal(EM.finish_forward(z.detach(), x.detach()), y.detach())
    gy = torch.randn(n, t, v, d, generator=g, dtype=torch.float64)
    gz_r, gx_r = torch.autograd.grad(y, (z, x), gy)
    gz, gx = EM.finish_backward(gy, True)
    assert max_abs(gz, gz_r) < 1e-13 and max_abs(gx, gx_r) < 1e-13
    pred = torch.randn(n, t, v * d, generator=g, dtype=torch.float64, requires_grad=True)
    tgt = torch.randn(n, t, v * d, generator=g, dtype=torch.float64)
    loss = pose_loss(pred, tgt, d) * 0.5
    (gp_r,) = torch.autograd.grad(loss, pred)
    acc = torch.full((), 2.0, dtype=torch.float64)
    gp = EM.pose_error(pred.detach(), tgt, 0.5, acc, True, d)
    assert abs(float(acc) - 2.0 - float(loss.detach())) < 1e-14 and max_abs(gp, gp_r) < 1e-15


@pytest.fixture
def dims_backend():
    prev = _lib._set_backend_for_tests(EM)
    yield
    _lib._set_backend_for_tests(prev)


@pytest.mark.parametrize("variant", ["std", "fast"])
def test_model_at_2_coordinates_through_host_wiring(variant, dims_backend):
    """A D = 2 model (input_channels = 4) through modules -> autograd -> ops on the fp64 emulation, against autograd of
    the oracle network with the restated head and tail."""
    fast = variant == "fast"
    torch.manual_seed(3)
    m = _perturbed(_mod(variant).DSTDGCN(4, 4, 6, 0.0, 22, 8, 2, "h36m")).double().train()
    assert m.coords == 2 and m.conv_st_out.stgcn[0][0].conv_t[0].out_channels == 2
    p = orc.state_from_module(m, torch.float64)
    x = torch.randn(3, 10, 22, 2, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    xr = x.clone().requires_grad_(True)
    yr = orc.dstdgcn(xr, p, True, fast)
    yr.pow(2).mean().backward()
    xm = x.clone().requires_grad_(True)
    y = m(xm)
    y.pow(2).mean().backward()
    assert y.shape == x.shape and max_abs(y, yr) < 1e-9
    assert rel_err(xm.grad, xr.grad) < 1e-9
    for k, prm in m.named_parameters():
        if prm.grad is not None:
            assert max_abs(prm.grad, p[k].grad) < 1e-8 * max(1.0, float(p[k].grad.abs().max())), k


def test_train_step_at_2_coordinates_on_emulation(dims_backend):
    """TrainStep on [N, T, 2V] batches reads D from the model; its loss is the restated one."""
    torch.manual_seed(5)
    m = _perturbed(_mod("std").DSTDGCN(4, 4, 6, 0.0, 22, 8, 1, "h36m")).double().train()
    p = orc.state_from_module(m, torch.float64)
    g = torch.Generator().manual_seed(6)
    a = torch.randn(2, 10, 44, generator=g, dtype=torch.float64)
    tg = a + 0.1 * torch.randn(2, 10, 44, generator=g, dtype=torch.float64)
    b = torch.flip(a, dims=[1]).contiguous()
    ref = train_loss(p, a, b, tg, 2)
    step = engine.TrainStep(m, lr=3e-3, inverse=True)
    assert abs(float(step(a, b, tg)) - float(ref)) < 1e-6 * float(ref)       # the loss scalar is fp32
    pred = engine.predict(m, a)
    assert pred.shape == a.shape


@pytest.mark.parametrize("cin,d,exc,match", [
    (5, 2, ValueError, "input_channels = 5"),
    (5, 3, ValueError, "input_channels = 5"),
    (4, 3, ValueError, r"input_channels = 4 .* = 2 coordinates per joint; x has 3"),
    (6, 2, ValueError, r"input_channels = 6 .* = 3 coordinates per joint; x has 2"),
    (66, 33, NotImplementedError, "at most 32 coordinates"),
])
def test_input_validation(cin, d, exc, match, dims_backend):
    m = _mod("std").DSTDGCN(cin, 2, 2, 0.0, 22, 8, 1, "h36m")
    with pytest.raises(exc, match=match):
        m(torch.zeros(1, 4, 22, d))


def test_mirror_and_window_batch_at_2_coordinates():
    rng = np.random.default_rng(12)
    a = rng.standard_normal((3, 35, 32 * 2)).astype(np.float32)
    src = a.reshape(3, 35, 32, 2)
    ref = src.copy()
    ref[:, :, data._H36M_RIGHT] = src[:, :, data._H36M_LEFT]
    ref[:, :, data._H36M_LEFT] = src[:, :, data._H36M_RIGHT]
    ref[..., 0] = -ref[..., 0]
    got = data.mirror(torch.from_numpy(a), "h36m", dims=2)
    assert np.array_equal(got.numpy(), ref.reshape(3, 35, 64))
    assert np.array_equal(data.mirror(got, "h36m", dims=2).numpy(), a)
    used = np.setdiff1d(np.arange(64), np.concatenate([np.array([0, 1, 6, 11, 16, 20, 23, 24, 28, 31]) * 2 + c
                                                       for c in range(2)]))
    i_idx = np.append(np.arange(0, 10), np.repeat([9], 25))
    i_inv = np.append(np.arange(25, 35)[::-1], np.repeat([25], 25))
    for (x, r) in zip(data.window_batch(torch.from_numpy(a), 10, 25, used),
                      (a[:, i_idx][:, :, used], a[:, i_inv][:, :, used], a[:, :, used])):
        assert np.array_equal(x.numpy(), r)
    (b,) = list(data.DevicePrefetcher([a], 10, 25, used, device="cpu", mirror_layout="h36m", dims=2))
    assert np.array_equal(b[3].numpy(), np.concatenate((a, ref.reshape(3, 35, 64))))


class _Shift2(torch.nn.Module):
    """Stand-in model on 2-D joints: [N,T,V,2] -> same shape."""
    coords = 2

    def forward(self, x):
        assert x.shape[-1] == 2
        return x * 0.9 + 0.05


def test_evaluate_at_2_coordinates():
    """engine.evaluate against the reference lines (engine/prediction.py:366-406) with 2 columns per joint."""
    g = torch.Generator().manual_seed(8)
    joints_full, t_all, input_n, d = 32, 35, 10, 2
    used_j = np.array([j for j in range(joints_full) if j not in (0, 1, 6, 11, 16, 20, 23, 24, 28, 31)])
    dim_used = np.sort(np.concatenate([used_j * d + c for c in range(d)]))
    ign, eq = np.array([16, 20, 23, 24, 28, 31]), np.array([13, 19, 22, 13, 27, 30])
    eval_frame = [1, 3, 7, 9, 13, 24]
    batches = []
    for n in (5, 3):
        seqs = torch.randn(n, t_all, joints_full * d, generator=g)
        batches.append((seqs[:, :, dim_used].clone(), seqs))
    model = _Shift2()
    avg, per_frame = engine.evaluate(model, batches, input_n, eval_frame, dim_used, ign, eq)
    tot, acc, cnt_all, n_tot = np.zeros(len(eval_frame)), 0.0, 0, 0
    for inputs, seqs in batches:
        n = inputs.shape[0]
        out = model(inputs.view(n, t_all, -1, d)).reshape(n, t_all, -1).numpy()
        pred = seqs.numpy().copy()
        pred[:, :, dim_used] = out
        i_ign = np.concatenate([ign * d + c for c in range(d)])
        i_eq = np.concatenate([eq * d + c for c in range(d)])
        pred[:, :, i_ign] = pred[:, :, i_eq]
        p3 = pred.reshape(n, t_all, -1, d)[:, input_n:]
        t3 = seqs.numpy().reshape(n, t_all, -1, d)[:, input_n:]
        for k, j in enumerate(eval_frame):
            e = np.mean(np.linalg.norm(t3[:, j].reshape(-1, d) - p3[:, j].reshape(-1, d), axis=1)) * n
            tot[k] += e
            acc += e
            cnt_all += n
        n_tot += n
    assert np.allclose(per_frame, tot / n_tot, rtol=1e-5, atol=1e-6)
    assert abs(avg - acc / cnt_all) < 1e-5


_CTYPE = {"int": ctypes.c_int, "float": ctypes.c_float, "long long": ctypes.c_longlong, "size_t": ctypes.c_size_t,
          "dstd_view": _lib.View, "dstd_stream_t": ctypes.c_void_p}
NEW_SYMBOLS = ["dstd_prep_forward_d", "dstd_prep_backward_d", "dstd_finish_forward_d", "dstd_finish_backward_d",
               "dstd_pose_error_workspace_bytes", "dstd_pose_error_forward_backward"]


@pytest.mark.parametrize("name", NEW_SYMBOLS)
def test_new_prototypes_match_header(name):
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "dstd_b200.h")).read(), flags=re.S)
    ret, params = re.search(r"(\w+)\s+" + name + r"\(([^)]*)\);", src).groups()

    def ctype(decl):
        decl = decl.strip()
        if "*" in decl:
            return ctypes.c_void_p
        return _CTYPE[" ".join(decl.replace("const ", "").split()[:-1])]

    res, args = _lib.SYMBOLS[name]
    assert res is _CTYPE[ret]
    assert args == [ctype(p) for p in params.split(",")]


# ====================================================================================================== GPU
def _be():
    b = _lib.backend()
    assert b.name == "cuda"
    return b


def _to_dev(t):
    out = torch.empty_strided(t.shape, t.stride(), dtype=torch.float32, device=DEV)
    out.copy_(t.float())
    return out


def _nctv(g, n, c, t, v, order):
    """Logical [N,C,T,V] fp64 tensor in T-major, V-major or the fast variant's [N,T,V,C] memory order."""
    if order == "t":
        return torch.randn((n, c, t, v), generator=g, dtype=torch.float64)
    if order == "v":
        return torch.randn((n, c, v, t), generator=g, dtype=torch.float64).permute(0, 1, 3, 2)
    return torch.randn((n, t, v, c), generator=g, dtype=torch.float64).permute(0, 3, 1, 2)


def _empty_like_order(n, c, t, v, order):
    return _to_dev(_nctv(torch.Generator().manual_seed(0), n, c, t, v, order)).fill_(float("nan"))


def _call(fn, *args):
    lib = _be().lib
    rc = getattr(lib, fn)(*args, None)
    assert rc == 0, (fn, lib.dstd_last_error())


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _v(t):
    s = t.stride()
    return _lib.View(ctypes.c_void_p(t.data_ptr()), *s)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 2, 4, 32])
@pytest.mark.parametrize("order", ["t", "v", "fast"])
@pytest.mark.parametrize("n,t,v", [(3, 7, 5), (2, 35, 22)])
def test_entry_points_vs_emulation(d, order, n, t, v):
    g = torch.Generator().manual_seed(d * 100 + n * t + v)
    x = torch.randn(n, t, v, d, generator=g, dtype=torch.float64)
    xd = _to_dev(x)
    # prep forward / backward
    h = _empty_like_order(n, 2 * d, t, v, order)
    _call("dstd_prep_forward_d", _p(xd), _v(h), n, t, v, d)
    assert max_abs(h, EM.prep_forward(x)) < 1e-6
    gh = _nctv(g, n, 2 * d, t, v, order)
    ghd = _to_dev(gh)
    gx = torch.full((n, t, v, d), float("nan"), device=DEV)
    _call("dstd_prep_backward_d", _v(ghd), _p(gx), n, t, v, d)
    assert max_abs(gx, EM.prep_backward(gh)) < 1e-5
    # finish forward / backward, gx wanted and not
    z = _nctv(g, n, d, t, v, order)
    zd = _to_dev(z)
    y = torch.full((n, t, v, d), float("nan"), device=DEV)
    _call("dstd_finish_forward_d", _v(zd), _p(xd), _p(y), n, t, v, d)
    assert max_abs(y, EM.finish_forward(z, x)) < 1e-6
    gy = torch.randn(n, t, v, d, generator=g, dtype=torch.float64)
    gz_r, gx_r = EM.finish_backward(gy, True)
    gyd = _to_dev(gy)
    for want_gx in (True, False):
        gz = _empty_like_order(n, d, t, v, order)
        gx = torch.full((n, t, v, d), float("nan"), device=DEV) if want_gx else None
        _call("dstd_finish_backward_d", _p(gyd), _v(gz), _p(gx), n, t, v, d)
        assert max_abs(gz, gz_r) < 1e-6
        if want_gx:
            assert max_abs(gx, gx_r) < 1e-5
    # loss: scale, accumulate, repeat call
    pred, tgt = torch.randn(n, t, v * d, generator=g, dtype=torch.float64), torch.randn(n, t, v * d, generator=g,
                                                                                          dtype=torch.float64)
    l_r = torch.zeros((), dtype=torch.float64)
    gp_r = EM.pose_error(pred, tgt, 0.5, l_r, False, d)
    be = _be()
    pd_, td = _to_dev(pred), _to_dev(tgt)
    loss = torch.zeros((), device=DEV)
    gp = be.pose_error(pd_, td, 0.5, loss, False, d)
    torch.cuda.synchronize()
    assert abs(float(loss) - float(l_r)) < 2e-6 * max(1.0, float(l_r)) and max_abs(gp, gp_r) < 1e-8
    loss2 = torch.full((), 0.25, device=DEV)
    gp2 = be.pose_error(pd_, td, 0.5, loss2, True, d)
    assert abs(float(loss2) - 0.25 - float(l_r)) < 2e-6 * max(1.0, float(l_r))
    loss3 = torch.zeros((), device=DEV)
    gp3 = be.pose_error(pd_, td, 0.5, loss3, False, d)
    assert torch.equal(gp, gp2) and torch.equal(gp, gp3) and torch.equal(loss, loss3)


@pytest.mark.gpu
def test_entry_points_refuse_33_coordinates():
    lib = _be().lib
    x = torch.zeros(1, 2, 3, 33, device=DEV)
    h = torch.zeros(1, 66, 2, 3, device=DEV)
    assert lib.dstd_prep_forward_d(_p(x), _v(h), 1, 2, 3, 33, None) == -2
    assert b"1..32" in lib.dstd_last_error()
    ws = torch.empty(1 << 12, dtype=torch.uint8, device=DEV)
    loss = torch.zeros((), device=DEV)
    assert lib.dstd_pose_error_forward_backward(_p(x), _p(x), 6, 0, 1.0, 0, _p(loss), _p(x), _p(ws), ws.numel(),
                                                None) == -2
    assert b"1..32" in lib.dstd_last_error()


@pytest.mark.gpu
@pytest.mark.parametrize("order", ["t", "v", "fast"])
def test_d_entry_points_at_xyz_give_the_original_bits(order):
    g = torch.Generator().manual_seed(33)
    n, t, v, d = 37, 35, 22, 3
    xd = _to_dev(torch.randn(n, t, v, d, generator=g, dtype=torch.float64))
    outs = []
    for suffix, extra in (("", ()), ("_d", (d,))):
        h = _empty_like_order(n, 6, t, v, order)
        _call("dstd_prep_forward" + suffix, _p(xd), _v(h), n, t, v, *extra)
        gh = _to_dev(_nctv(torch.Generator().manual_seed(1), n, 6, t, v, order))
        gx = torch.empty(n, t, v, d, device=DEV)
        _call("dstd_prep_backward" + suffix, _v(gh), _p(gx), n, t, v, *extra)
        z = _to_dev(_nctv(torch.Generator().manual_seed(2), n, 3, t, v, order))
        y = torch.empty(n, t, v, d, device=DEV)
        _call("dstd_finish_forward" + suffix, _v(z), _p(xd), _p(y), n, t, v, *extra)
        gz, gx2 = _empty_like_order(n, 3, t, v, order), torch.empty(n, t, v, d, device=DEV)
        _call("dstd_finish_backward" + suffix, _p(y), _v(gz), _p(gx2), n, t, v, *extra)
        outs.append((h, gx, y, gz, gx2))
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    be = _be()
    pred = _to_dev(torch.randn(n, t, v * 3, generator=g, dtype=torch.float64))
    tgt = _to_dev(torch.randn(n, t, v * 3, generator=g, dtype=torch.float64))
    l1, l2 = torch.full((), 0.5, device=DEV), torch.full((), 0.5, device=DEV)
    g1 = be.mpjpe(pred, tgt, 0.5, l1, True)
    g2 = be.pose_error(pred, tgt, 0.5, l2, True, 3)
    assert torch.equal(g1, g2) and torch.equal(l1, l2)


def _model_check(variant, d, seed):
    """test_gpu_parity._full_size_check at D coordinates: the fp32 restatement (the reference's arithmetic) against fp64
    is the yardstick."""
    fast = variant == "fast"
    v, tin, tout = 22, 10, 25
    torch.manual_seed(777)
    m = _perturbed(_mod(variant).DSTDGCN(2 * d, tin, tout, 0.0, v, 64, 5, "h36m"))
    x = torch.randn(4, tin + tout, v, d, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)

    def run_oracle(dtype):
        p = orc.state_from_module(m, dtype)
        xx = x.to(dtype).clone().requires_grad_(True)
        y = orc.dstdgcn(xx, p, True, fast)
        y.pow(2).mean().backward()
        return y.detach(), xx.grad, {k: t.grad for k, t in p.items() if t.requires_grad and t.grad is not None}

    y64, gx64, g64 = run_oracle(torch.float64)
    y32, gx32, g32 = run_oracle(torch.float32)
    md = m.to(DEV).train()
    xd = x.float().to(DEV).requires_grad_(True)
    y = md(xd)
    y.pow(2).mean().backward()
    assert rel_err(y, y64) < 4 * rel_err(y32, y64)
    assert rel_err(xd.grad, gx64) < 3.5 * rel_err(gx32, gx64)
    num = den = num32 = 0.0
    for k, p in md.named_parameters():
        if p.grad is None:
            continue
        diff = p.grad.double().cpu() - g64[k]
        num += float((diff * diff).sum())
        num32 += float(((g32[k].double() - g64[k]) ** 2).sum())
        den += float((g64[k] ** 2).sum())
    rel, rel32 = (num / den) ** 0.5, (num32 / den) ** 0.5
    assert rel < 3.5 * rel32, (rel, rel32)
    gmax = max(float(t.abs().max()) for t in g64.values())
    bad = []
    for k, p in md.named_parameters():
        if p.grad is None:
            continue
        e, e32, scale = max_abs(p.grad, g64[k]), max_abs(g32[k], g64[k]), float(g64[k].abs().max())
        if e > max(10 * e32, 8e-2 * scale, 2e-6 * gmax):
            bad.append((k, e, e32, scale))
    assert not bad, bad[:5]


@pytest.mark.gpu
@pytest.mark.parametrize("variant,d,seed", [("std", 2, 1234), ("fast", 2, 11), ("std", 4, 1234), ("fast", 4, 1234)])
def test_model_vs_restatement(variant, d, seed):
    """As in test_custom_skeleton.py::test_model_vs_oracle_wide, an input at which a pre-activation sits on a PReLU kink
    within rounding distance makes either side's dx, or a PReLU-slope gradient, jump by 1e-3 .. 1e-2.  The fast
    variant meets such inputs at every D, the unchanged xyz path included: its dx error over the fp32 restatement's is
    1.4 .. 4.7 at D = 3 and 0.4 .. 79 at D = 4 across seeds 1234, 99, 7, 5, while y stays at 3.1 .. 3.6 everywhere.  The
    fast D = 2 case uses seed 11, which is not at such a point (1234, 99, 42, 77, 123 are; 21 and 2024 are not)."""
    _model_check(variant, d, seed)


def _batches(n, v, d, steps, seed):
    """[N, 35, D*V] random-walk windows: (inputs, inputs_inv, targets) as bench.synthetic_batch builds them for xyz."""
    out = []
    for s in range(steps):
        g = torch.Generator().manual_seed(seed + s)
        seq = torch.randn(n, 1, v * d, generator=g) + torch.cumsum(torch.randn(n, 35, v * d, generator=g) * 0.05, dim=1)
        fwd, inv = data.window_indices(10, 25)
        out.append((seq[:, fwd].contiguous(), seq[:, inv].contiguous(), seq.contiguous()))
    return out


@pytest.mark.gpu
def test_train_steps_at_2_coordinates_vs_restatement():
    """Three Adam steps of DSTDGCN(4, 10, 25, 0.1, 22, 64, 5) through TrainStep on [256, 35, 44] batches, with the same
    dropout masks as the restatement, gated like the full-size dropout test of test_gpu_parity.py at its batch; then
    engine.evaluate scores the trained model.  Adam turns rounding-level gradient differences into +-lr moves, so the
    gate follows how fast the fp32 restatement separates from fp64.  The batches of seed 500 sit on the gate's 1e-3
    floor at the second step (1.1e-3 here, 2.5e-4 for the fp32 restatement; 6.6e-3 and 2.3e-2 at the third); seeds
    600, 700 and 800 pass."""
    _train_check(600)


def _train_check(seed):
    n, v, c, drop, steps, d = 256, 22, 64, 0.1, 3, 2
    torch.manual_seed(777)
    m = _perturbed(_mod("std").DSTDGCN(2 * d, 10, 25, drop, v, c, 5, "h36m"))
    g = torch.Generator().manual_seed(99)
    masks = [[(torch.rand(n, c, 35, v, generator=g) >= drop).float() / (1.0 - drop) for _ in range(2)]
             for _ in range(steps)]
    batches = _batches(n, v, d, steps, seed)

    def trajectory(dtype):
        p = orc.state_from_module(m, dtype)
        opt = torch.optim.Adam([x for x in p.values() if x.requires_grad], lr=3e-3)
        out = []
        for s in range(steps):
            a, b, tg = (x.to(dtype) for x in batches[s])
            loss = train_loss(p, a, b, tg, d, dropout_masks=tuple(mk.to(dtype) for mk in masks[s]))
            opt.zero_grad()
            loss.backward()
            opt.step()
            out.append(float(loss.detach()))
        return out

    ref, ref32 = trajectory(torch.float64), trajectory(torch.float32)
    md = m.to(DEV).train()
    step = engine.TrainStep(md, lr=3e-3, inverse=True)
    got = []
    for s in range(steps):
        md.dropout_mask = [mk.to(DEV) for mk in masks[s]]
        md._mask_calls = 0
        got.append(float(step(*(x.to(DEV) for x in batches[s]))))
    ref_t, got_t, r32_t = (torch.tensor(x, dtype=torch.float64) for x in (ref, got, ref32))
    dev, dev32 = (got_t - ref_t).abs() / ref_t.abs(), (r32_t - ref_t).abs() / ref_t.abs()
    assert float(dev[0]) < 1e-4, (got, ref)
    assert bool((dev <= torch.clamp(4 * dev32, min=1e-3)).all()), (got, ref, ref32)
    md.dropout_mask = None
    seqs = batches[0][2].to(DEV)
    avg, per_frame = engine.evaluate(md, [(seqs, seqs)], 10, [1, 9, 24])
    assert md.training and np.isfinite(avg) and per_frame.shape == (3,)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["std", "fast"])
def test_captured_step_equals_eager_at_2_coordinates(variant):
    batches = [tuple(x.to(DEV) for x in b) for b in _batches(16, 22, 2, 3, 40)]

    def fresh():
        torch.manual_seed(5)
        m = _perturbed(_mod(variant).DSTDGCN(4, 10, 25, 0.0, 22, 16, 2, "h36m")).to(DEV).train()
        return m, engine.TrainStep(m, lr=3e-3, inverse=True)

    m_a, st_a = fresh()
    la = [float(st_a(*b)) for b in batches]
    m_b, st_b = fresh()
    st_b.capture(*batches[0])
    lb = [float(st_b(*b)) for b in batches]
    assert st_b.graph is not None
    assert max(abs(a - b) for a, b in zip(la, lb)) < 1e-6
    sa, sb = m_a.state_dict(), m_b.state_dict()
    for k in sa:
        assert max_abs(sa[k], sb[k]) < 1e-6, k


def step_kernels(d):
    """Library kernels launched by one eager TrainStep (both passes on one stream, so the order is fixed) of
    DSTDGCN(2D, 10, 25, 0.1, 22, 16, 2), in launch order, names cut at '<' / '(' and without 'dstd::'.

    The profiler can miss the first kernels after it starts when it has run earlier in the process (in the full suite
    it dropped the first 8 of 257), so two steps are profiled and the kernels of the second are taken: as many as the
    library counts for one step (dstd_kernel_launch_count)."""
    from torch.profiler import ProfilerActivity, profile
    torch.manual_seed(3)
    m = _perturbed(_mod("std").DSTDGCN(2 * d, 10, 25, 0.1, 22, 16, 2, "h36m")).to(DEV).train()
    step = engine.TrainStep(m, lr=3e-3, inverse=True)
    step._overlap = False
    b = tuple(x.to(DEV) for x in _batches(8, 22, d, 1, 7)[0])
    be = _be()
    step(*b)                                          # warm-up
    torch.cuda.synchronize()
    l0 = be.launches
    step(*b)
    torch.cuda.synchronize()
    per_step = be.launches - l0
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step(*b)
        step(*b)
        torch.cuda.synchronize()
    evs = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "dstd::" in e.name),
                 key=lambda e: e.time_range.start)
    names = [e.name.removeprefix("void ").removeprefix("dstd::").split("(")[0].split("<")[0] for e in evs]
    assert per_step <= len(names) <= 2 * per_step, (per_step, len(names))
    return names[-per_step:]


def _first_diff(got, want):
    """Where two launch lists part: index, lengths and a window of both."""
    i = next((i for i, (a, b) in enumerate(zip(got, want)) if a != b), min(len(got), len(want)))
    return f"first difference at {i} of {len(got)} / {len(want)}: {got[max(0, i - 3):i + 6]} vs {want[max(0, i - 3):i + 6]}"


def _expand(table):
    out = []
    for tok in table.split():
        name, _, k = tok.partition("*")
        out += [name + "_kernel"] * int(k or 1)
    return out


# step_kernels(3) recorded with the library of the commit before the D-generic heads (names without `_kernel`;
# `name*k` = k consecutive launches).  The xyz step must launch exactly this.
XYZ_STEP_KERNELS = (
    "prep_fwd bgemm bn_stats bnf_apply pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc bn_stats bnf_apply "
    "pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc bn_stats bn_apply pack mproj_fwd dynadj_fwd_mma pack_tc "
    "aggmix_fwd_tc bn_stats bnf_apply pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc bn_stats bnf_apply pack "
    "mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc bn_stats bnf_apply pack mproj_fwd dynadj_fwd_mma pack_tc "
    "aggmix_fwd_tc bn_stats bnf_apply bgemm bn_stats bn_apply pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc "
    "bn_stats bn_apply pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc finish_fwd mpjpe mpjpe_finish "
    "finish_bwd pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments bn_bwd_reduce bn_bwd_apply pack "
    "aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments bn_bwd_reduce bn_bwd_apply bgemm wgrad reduce_segments "
    "bnf_bwd_reduce bnf_bwd_apply pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments bnf_bwd_reduce "
    "bnf_bwd_apply pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments bnf_bwd_reduce bnf_bwd_apply pack "
    "aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments bnf_bwd_reduce bnf_bwd_apply pack aggmix_bwd "
    "dynadj_bwd_mma mproj_bwd reduce_segments bn_bwd_reduce bn_bwd_apply pack aggmix_bwd dynadj_bwd_mma mproj_bwd "
    "reduce_segments bnf_bwd_reduce bnf_bwd_apply pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments "
    "bnf_bwd_reduce bnf_bwd_apply wgrad reduce_segments prep_fwd bgemm bn_stats bnf_apply pack mproj_fwd "
    "dynadj_fwd_mma pack_tc aggmix_fwd_tc bn_stats bnf_apply pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc "
    "bn_stats bn_apply pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc bn_stats bnf_apply pack mproj_fwd "
    "dynadj_fwd_mma pack_tc aggmix_fwd_tc bn_stats bnf_apply pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc "
    "bn_stats bnf_apply pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc bn_stats bnf_apply bgemm bn_stats "
    "bn_apply pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc bn_stats bn_apply pack mproj_fwd dynadj_fwd_mma "
    "pack_tc aggmix_fwd_tc finish_fwd mpjpe mpjpe_finish finish_bwd pack aggmix_bwd dynadj_bwd_mma mproj_bwd "
    "reduce_segments bn_bwd_reduce bn_bwd_apply pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments "
    "bn_bwd_reduce bn_bwd_apply bgemm wgrad reduce_segments bnf_bwd_reduce bnf_bwd_apply pack aggmix_bwd "
    "dynadj_bwd_mma mproj_bwd reduce_segments bnf_bwd_reduce bnf_bwd_apply pack aggmix_bwd dynadj_bwd_mma "
    "mproj_bwd reduce_segments bnf_bwd_reduce bnf_bwd_apply pack aggmix_bwd dynadj_bwd_mma mproj_bwd "
    "reduce_segments bnf_bwd_reduce bnf_bwd_apply pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments "
    "bn_bwd_reduce bn_bwd_apply pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments bnf_bwd_reduce "
    "bnf_bwd_apply pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments bnf_bwd_reduce bnf_bwd_apply wgrad "
    "reduce_segments adam ")


@pytest.mark.gpu
def test_step_launches():
    """D = 3 launches what it launched before D-generic heads existed.  D = 2 launches the same list with the
    D-generic head, tail and loss kernels in place of the xyz ones; the only other difference is the path of the two
    BatchNorms over the last layer's D channels: the bulk-copy kernels take a 2-channel plane at H3.6M, the generic
    ones a 3-channel one (the unchanged slab rule; the two paths are bit-identical)."""
    xyz, two = step_kernels(3), step_kernels(2)
    assert xyz == _expand(XYZ_STEP_KERNELS), _first_diff(xyz, _expand(XYZ_STEP_KERNELS))
    swap = {"prep_fwd_kernel": "prep_fwd_d_kernel", "finish_fwd_kernel": "finish_fwd_d_kernel",
            "finish_bwd_kernel": "finish_bwd_d_kernel", "mpjpe_kernel": "pose_error_kernel"}
    assert all(xyz.count(k) == 2 for k in swap) and not set(swap.values()) & set(xyz)       # one per pass
    # the batch needs no input gradient, so neither prep backward runs
    assert "prep_bwd_kernel" not in xyz and "prep_bwd_d_kernel" not in two
    same_bn_path = lambda ks: [k.replace("bnf_", "bn_") for k in ks]
    assert same_bn_path(two) == same_bn_path([swap.get(k, k) for k in xyz]), _first_diff(two, xyz)
    changed = [(a, b) for a, b in zip([swap.get(k, k) for k in xyz], two) if a != b]
    assert len(changed) == 12 and all(b == a.replace("bn_", "bnf_") for a, b in changed), changed
