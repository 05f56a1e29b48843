"""`torch.library` operators (namespace ``dstd_b200``) over the C ABI, and their autograd wiring.

Layering:  nn.Module mirrors (model/)  ->  functions in this file (autograd.Function)
           ->  ``torch.ops.dstd_b200.*`` custom ops  ->  ``_lib.backend()`` (ctypes -> libdstd_b200.so).

The custom ops are registered for CUDA only; there is no CPU kernel, so calling
them with CPU tensors raises (the test-suite swaps in the ABI emulation from
``oracle/`` explicitly to exercise this wiring without a GPU).
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import os

import torch
import torch.distributed as dist
from torch import Tensor

from . import _lib

_BR_KEYS = ("w_m1", "b_m1", "w_m2", "b_m2", "w_rm", "b_rm", "w_f", "b_f", "adj", "adj_w", "adj_r")
_NBK = len(_BR_KEYS)
_GR_KEYS = ("w_m1", "b_m1", "w_m2", "b_m2", "w_rm", "b_rm", "w_f", "b_f")

_DEV = None  # custom ops are device-agnostic at registration; the backend enforces CUDA tensors


def _unflatten(flat: Sequence[Optional[Tensor]], nb: int):
    return [{k: flat[b * _NBK + i] for i, k in enumerate(_BR_KEYS)} for b in range(nb)]


ORDER_LIKE_INPUT, ORDER_T_MAJOR, ORDER_V_MAJOR = 0, 1, 2


def _out_like(y: Tensor, order: int) -> Tensor:
    """Stride template for a logical [N,C,T,V] output: like y, [N,C,T,V]-contiguous, or [N,C,V,T]-contiguous.
    Returned tensor shares no storage semantics with the result (expanded 1-element dummy)."""
    if order == ORDER_LIKE_INPUT:
        return y
    n, c, t, v = y.shape
    strides = (c * t * v, t * v, v, 1) if order == ORDER_T_MAJOR else (c * t * v, t * v, 1, t)
    return torch.empty_strided((n, c, t, v), strides, dtype=y.dtype, device="meta")


# =========================================================================== custom ops
@torch.library.custom_op("dstd_b200::gc_fwd", mutates_args=())
def gc_fwd(x: Tensor, alpha: Optional[Tensor], br: Sequence[Optional[Tensor]], skip: Optional[Tensor], nb: int,
           adj_t: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    return _lib.backend().gc_forward(x, alpha, _unflatten(br, nb), skip, adj_t)


@gc_fwd.register_fake
def _(x, alpha, br, skip, nb, adj_t):
    n, cin, p, k = x.shape
    cout = br[6].shape[0]
    need_xa = bool(_lib.load_library().dstd_gc_needs_xa(cin, cout, p, k, nb))
    return (_lib._like_layout(x, cout), x.new_empty((n, nb, 4, p, k)), x.new_empty((n, nb, p, k, k)),
            x.new_empty((n, nb, cin + 1, p, k) if need_xa else (0,)))


@torch.library.custom_op("dstd_b200::gc_bwd", mutates_args=())
def gc_bwd(x: Tensor, gout: Tensor, alpha: Optional[Tensor], br: Sequence[Optional[Tensor]], m: Tensor, pd: Tensor,
           xa: Tensor, nb: int, adj_t: bool, gx_add: Optional[Tensor] = None) -> List[Tensor]:
    """Returns [gx (+ gx_add), galpha, then per branch: 8 weight grads, adj_eff grad, adj_w grad]; unused slots are
    0-size."""
    brs = _unflatten(br, nb)
    gx, galpha, grads = _lib.backend().gc_backward(x, gout, alpha, brs, m, pd, xa, adj_t, True, gx_add)
    out = [gx, galpha if galpha is not None else x.new_empty((0,))]
    for g in grads:
        out += [g[k] for k in _GR_KEYS] + [g["adj_eff"], g["adj_w"] if g["adj_w"] is not None else x.new_empty((0,))]
    return out


@gc_bwd.register_fake
def _(x, gout, alpha, br, m, pd, xa, nb, adj_t, gx_add=None):
    k = x.shape[3]
    out = [torch.empty_like(x), x.new_empty((1,) if alpha is not None else (0,))]
    for b in range(nb):
        out += [torch.empty_like(br[b * _NBK + i]) for i in range(8)]
        out += [x.new_empty((k, k)), x.new_empty((k, k) if br[b * _NBK + 9] is not None else (0,))]
    return out


@torch.library.custom_op("dstd_b200::bn_act_fwd", mutates_args=("running_mean", "running_var", "nbt"))
def bn_act_fwd(y: Tensor, r: Optional[Tensor], gamma: Tensor, beta: Tensor, running_mean: Optional[Tensor],
               running_var: Optional[Tensor], nbt: Optional[Tensor], prelu: Optional[Tensor], mask: Optional[Tensor],
               out_order: int, vc_order: bool, training: bool, eps: float,
               momentum: float) -> Tuple[Tensor, Tensor, Tensor]:
    return _lib.backend().bn_act_forward(y, r, gamma, beta, running_mean, running_var, nbt, prelu, mask, vc_order,
                                         training, eps, momentum, _out_like(y, out_order))


@bn_act_fwd.register_fake
def _(y, r, gamma, beta, running_mean, running_var, nbt, prelu, mask, out_order, vc_order, training, eps, momentum):
    return torch.empty_like(_out_like(y, out_order)), torch.empty_like(gamma), torch.empty_like(gamma)


@torch.library.custom_op("dstd_b200::bn_act_bwd", mutates_args=())
def bn_act_bwd(y: Tensor, r: Optional[Tensor], gout: Tensor, gamma: Tensor, beta: Tensor, prelu: Optional[Tensor],
               mask: Optional[Tensor], save_mean: Tensor, save_invstd: Tensor, vc_order: bool, training: bool,
               need_gr: bool, gr_add: Optional[Tensor] = None) -> List[Tensor]:
    """[gy, gr (+ gr_add)|empty, ggamma, gbeta, gprelu|empty]"""
    gy, gr, gg, gb, gp = _lib.backend().bn_act_backward(y, r, gout, gamma, beta, prelu, mask, save_mean, save_invstd,
                                                        vc_order, training, need_gr, gr_add)
    return [gy, gr if gr is not None else y.new_empty((0,)), gg, gb, gp if gp is not None else y.new_empty((0,))]


@bn_act_bwd.register_fake
def _(y, r, gout, gamma, beta, prelu, mask, save_mean, save_invstd, vc_order, training, need_gr, gr_add=None):
    return [torch.empty_like(y), torch.empty_like(r) if (r is not None and need_gr) else y.new_empty((0,)),
            torch.empty_like(gamma), torch.empty_like(gamma), y.new_empty((1,) if prelu is not None else (0,))]


# synchronised BatchNorm: each direction in two phases around an all-gather of fp64 rows (see sync_batch_norm)
@torch.library.custom_op("dstd_b200::bn_act_fwd_local", mutates_args=())
def bn_act_fwd_local(y: Tensor, vc_order: bool) -> Tensor:
    """This rank's exchange rows (count, mean, M2) [3*C*V] fp64."""
    return _lib.backend().bn_act_forward_local(y, vc_order)


@bn_act_fwd_local.register_fake
def _(y, vc_order):
    return y.new_empty((3 * y.shape[1] * y.shape[3],), dtype=torch.float64)


@torch.library.custom_op("dstd_b200::bn_act_fwd_global", mutates_args=("running_mean", "running_var", "nbt"))
def bn_act_fwd_global(y: Tensor, r: Optional[Tensor], gamma: Tensor, beta: Tensor, running_mean: Optional[Tensor],
                      running_var: Optional[Tensor], nbt: Optional[Tensor], prelu: Optional[Tensor],
                      mask: Optional[Tensor], all_rows: Tensor, out_order: int, vc_order: bool, eps: float,
                      momentum: float) -> Tuple[Tensor, Tensor, Tensor]:
    return _lib.backend().bn_act_forward_global(y, r, gamma, beta, running_mean, running_var, nbt, prelu, mask,
                                                vc_order, eps, momentum, all_rows, _out_like(y, out_order))


@bn_act_fwd_global.register_fake
def _(y, r, gamma, beta, running_mean, running_var, nbt, prelu, mask, all_rows, out_order, vc_order, eps, momentum):
    return torch.empty_like(_out_like(y, out_order)), torch.empty_like(gamma), torch.empty_like(gamma)


@torch.library.custom_op("dstd_b200::bn_act_bwd_local", mutates_args=())
def bn_act_bwd_local(y: Tensor, r: Optional[Tensor], gout: Tensor, gamma: Tensor, beta: Tensor,
                     prelu: Optional[Tensor], mask: Optional[Tensor], save_mean: Tensor, save_invstd: Tensor,
                     vc_order: bool, need_gr: bool, gr_add: Optional[Tensor] = None) -> List[Tensor]:
    """[ggamma, gbeta, gprelu|empty, exchange rows (count, sum g', sum g' xhat) [3*C*V] fp64, gy, gr|empty]; gy and
    gr are uninitialised buffers that bn_act_bwd_global fills."""
    gg, gb, gp, rows, gy, gr = _lib.backend().bn_act_backward_local(y, r, gout, gamma, beta, prelu, mask, save_mean,
                                                                    save_invstd, vc_order, need_gr, gr_add)
    return [gg, gb, gp if gp is not None else y.new_empty((0,)), rows, gy, gr if gr is not None else y.new_empty((0,))]


@bn_act_bwd_local.register_fake
def _(y, r, gout, gamma, beta, prelu, mask, save_mean, save_invstd, vc_order, need_gr, gr_add=None):
    return [torch.empty_like(gamma), torch.empty_like(gamma), y.new_empty((1,) if prelu is not None else (0,)),
            y.new_empty((3 * gamma.numel(),), dtype=torch.float64), torch.empty_like(y),
            torch.empty_like(r) if (r is not None and need_gr) else y.new_empty((0,))]


@torch.library.custom_op("dstd_b200::bn_act_bwd_global", mutates_args=("gy", "gr"))
def bn_act_bwd_global(y: Tensor, r: Optional[Tensor], gout: Tensor, gamma: Tensor, beta: Tensor,
                      prelu: Optional[Tensor], mask: Optional[Tensor], save_mean: Tensor, save_invstd: Tensor,
                      all_rows: Tensor, vc_order: bool, gy: Tensor, gr: Optional[Tensor],
                      gr_add: Optional[Tensor] = None) -> None:
    """Fills gy and gr (+ gr_add) (the buffers bn_act_bwd_local returned; gr None = not wanted)."""
    _lib.backend().bn_act_backward_global(y, r, gout, gamma, beta, prelu, mask, save_mean, save_invstd, vc_order,
                                          all_rows, gy, gr, gr_add)


@torch.library.custom_op("dstd_b200::chmix_fwd", mutates_args=())
def chmix_fwd(x: Tensor, w: Tensor, b: Optional[Tensor]) -> Tensor:
    return _lib.backend().chmix_forward(x, w, b)


@chmix_fwd.register_fake
def _(x, w, b):
    return _lib._like_layout(x, w.shape[0])


@torch.library.custom_op("dstd_b200::chmix_bwd", mutates_args=())
def chmix_bwd(x: Tensor, gout: Tensor, w: Tensor, need_gx: bool) -> List[Tensor]:
    gx, gw, gb = _lib.backend().chmix_backward(x, gout, w, need_gx)
    return [gx if gx is not None else x.new_empty((0,)), gw, gb]


@chmix_bwd.register_fake
def _(x, gout, w, need_gx):
    return [torch.empty_like(x) if need_gx else x.new_empty((0,)), torch.empty_like(w), x.new_empty((w.shape[0],))]


@torch.library.custom_op("dstd_b200::prep_fwd", mutates_args=())
def prep_fwd(x: Tensor) -> Tensor:
    return _lib.backend().prep_forward(x)


@prep_fwd.register_fake
def _(x):
    n, t, v, c = x.shape
    return x.new_empty((n, 2 * c, t, v))


@torch.library.custom_op("dstd_b200::prep_bwd", mutates_args=())
def prep_bwd(gh: Tensor) -> Tensor:
    return _lib.backend().prep_backward(gh)


@prep_bwd.register_fake
def _(gh):
    n, c, t, v = gh.shape
    return gh.new_empty((n, t, v, c // 2))


@torch.library.custom_op("dstd_b200::finish_fwd", mutates_args=())
def finish_fwd(z: Tensor, x: Tensor) -> Tensor:
    return _lib.backend().finish_forward(z, x)


@finish_fwd.register_fake
def _(z, x):
    return torch.empty_like(x)


@torch.library.custom_op("dstd_b200::finish_bwd", mutates_args=())
def finish_bwd(gy: Tensor, need_gx: bool) -> List[Tensor]:
    gz, gx = _lib.backend().finish_backward(gy, need_gx)
    return [gz, gx if gx is not None else gy.new_empty((0,))]


@finish_bwd.register_fake
def _(gy, need_gx):
    n, t, v, c = gy.shape
    return [gy.new_empty((n, c, t, v)), torch.empty_like(gy) if need_gx else gy.new_empty((0,))]


@torch.library.custom_op("dstd_b200::mpjpe", mutates_args=("loss",))
def mpjpe_op(pred: Tensor, target: Tensor, loss: Tensor, scale: float, accumulate: bool) -> Tensor:
    return _lib.backend().mpjpe(pred, target, scale, loss, accumulate)


@mpjpe_op.register_fake
def _(pred, target, loss, scale, accumulate):
    return torch.empty_like(pred)


@torch.library.custom_op("dstd_b200::adam_step", mutates_args=("param", "exp_avg", "exp_avg_sq"))
def adam_step(param: Tensor, grad: Tensor, exp_avg: Tensor, exp_avg_sq: Tensor, lr: float, beta1: float, beta2: float,
              eps: float, weight_decay: float, grad_scale: float, step: int, lr_dev: Optional[Tensor] = None,
              step_dev: Optional[Tensor] = None) -> None:
    _lib.backend().adam_step(param, grad, exp_avg, exp_avg_sq, lr, beta1, beta2, eps, weight_decay, grad_scale, step,
                             lr_dev, step_dev)


# =========================================================================== autograd
def _opt(t):
    return t if (t is not None and t.numel() > 0) else None


class _GcUnit(torch.autograd.Function):
    """Sum of `nb` DSTD-GC branches on unit coordinates [N,C,P,K] (+ optional skip)."""

    @staticmethod
    def forward(ctx, x, alpha, skip, nb, adj_t, pass_x, *flat):
        out, m, pd, xa = torch.ops.dstd_b200.gc_fwd(x, alpha, list(flat), skip, nb, adj_t)
        ctx.save_for_backward(x, alpha, m, pd, xa, *flat)
        ctx.nb, ctx.adj_t = nb, adj_t
        ctx.has_skip = skip is not None
        if pass_x:
            # second output = x itself: other consumers of x (the BN residual) use this alias, so their gradient comes
            # back through this node and is added by the kernel that writes gx (dstd_gc_bwd_args.gx_add)
            return out, x.view_as(x)
        return out

    @staticmethod
    def backward(ctx, gout, g_thru=None):
        x, alpha, m, pd, xa, *flat = ctx.saved_tensors
        nb = ctx.nb
        res = torch.ops.dstd_b200.gc_bwd(x, gout, alpha, list(flat), m, pd, xa, nb, ctx.adj_t, g_thru)
        gx, galpha = res[0], _opt(res[1])
        gflat = []
        for b in range(nb):
            g = res[2 + b * 10: 2 + (b + 1) * 10]
            adj, adj_w, adj_r = flat[b * _NBK + 8], flat[b * _NBK + 9], flat[b * _NBK + 10]
            geff, gadjw = g[8], _opt(g[9])
            gadj = None
            if ctx.needs_input_grad[6 + b * _NBK + 8]:
                gadj = geff if adj_w is None else geff * adj_w
            gflat += list(g[:8]) + [gadj, gadjw if adj_w is not None else None, geff if adj_r is not None else None]
        return (gx, galpha, gout if ctx.has_skip else None, None, None, None, *gflat)


def gc_unit(xu: Tensor, alpha: Optional[Tensor], branches: Sequence[dict], skip_u: Optional[Tensor] = None,
            adj_t: bool = False, pass_x: bool = False):
    """DSTD-GC unit.  ``xu``: [N,Cin,P,K] (any strides).  ``branches``: dicts with the keys of ``_BR_KEYS``
    (``adj_w``/``adj_r`` may be None/missing).  Returns [N,Cout,P,K] in the same memory order as ``xu``.
    ``pass_x``: also return ``xu`` as a second output of the same autograd node (see ``FUSE_SKIP_GRAD``)."""
    flat = []
    for br in branches:
        flat += [br.get(k) for k in _BR_KEYS]
    return _GcUnit.apply(xu, alpha, skip_u, len(branches), adj_t, bool(pass_x), *flat)


# The block input h feeds the spatial unit, the BN residual and the layer skip; autograd would sum the three gradients
# with two strided adds per block.  Instead the consumers are chained through pass-through outputs (h -> gc_unit
# (pass_x) -> bn_act residual (pass_r) -> skip), so the skip gradient is added inside the BN backward kernel
# (dstd_bn_act_bwd_args.gr_add) and the residual gradient inside the kernel that writes gx
# (dstd_gc_bwd_args.gx_add).  DSTD_FUSE_SKIP_GRAD=0 restores the plain autograd sums.
FUSE_SKIP_GRAD = os.environ.get("DSTD_FUSE_SKIP_GRAD", "1") not in ("", "0")
# the gx_add half of the chain is OFF by default: same-box A/B on B200 gave 9.30-9.43 k samples/s without any fusion,
# 9.53-9.59 k with the skip half only and 9.41-9.52 k with both (the extra read in the m-projection backward costs
# more than the strided add it removes)
FUSE_RES_GRAD = os.environ.get("DSTD_FUSE_RES_GRAD", "0") not in ("", "0")


# When a list, training-mode BatchNorm calls do NOT update their running statistics in the kernel; they append
# [running_mean, running_var, num_batches_tracked, momentum, eps, count, save_mean, save_invstd] instead and the caller
# applies the updates later with `apply_deferred_bn_updates` (engine.TrainStep runs the two passes of a step on two
# streams; the reference updates the statistics of the time-reversed pass AFTER those of the forward pass).
_bn_defer = None


class defer_bn_updates:
    """Context manager: collect the running-statistics updates of every BatchNorm call inside it."""

    def __init__(self):
        self.items = []

    def __enter__(self):
        global _bn_defer
        _refuse_sync_with_defer(_bn_sync)
        self._prev, _bn_defer = _bn_defer, self.items
        return self.items

    def __exit__(self, *exc):
        global _bn_defer
        _bn_defer = self._prev
        return False


@torch.no_grad()
def apply_deferred_bn_updates(items):
    """running = (1 - momentum) * running + momentum * batch statistic (unbiased variance), num_batches_tracked += 1
    (torch.nn.BatchNorm1d semantics, model/dstdgcn.py:42-49) for every collected call, in a handful of foreach kernels."""
    if not items:
        return
    groups = {}
    for rm, rv, nbt, mom, eps, cnt, mean, invstd in items:
        groups.setdefault((mom, eps, cnt), []).append((rm, rv, nbt, mean, invstd))
    for (mom, eps, cnt), g in groups.items():
        rms, rvs = [e[0] for e in g], [e[1] for e in g]
        nbts = [e[2] for e in g if e[2] is not None]
        means, invs = [e[3] for e in g], [e[4] for e in g]
        torch._foreach_mul_(rms, 1.0 - mom)
        torch._foreach_add_(rms, means, alpha=mom)
        var = torch._foreach_mul(invs, invs)
        torch._foreach_reciprocal_(var)                 # biased variance + eps
        torch._foreach_sub_(var, eps)
        torch._foreach_mul_(var, mom * (cnt / max(cnt - 1.0, 1.0)))
        torch._foreach_mul_(rvs, 1.0 - mom)
        torch._foreach_add_(rvs, var)
        if nbts:
            torch._foreach_add_(nbts, 1)


# When not None: the process group of the innermost active `sync_batch_norm` (a 1-tuple: the group may be None, the
# default group).
_bn_sync = None


def _sync_world(sync):
    return dist.get_world_size(sync[0]) if sync is not None and dist.is_available() and dist.is_initialized() else 1


def _refuse_sync_with_defer(sync):
    if _sync_world(sync) > 1:
        raise RuntimeError("sync_batch_norm cannot be combined with defer_bn_updates: synchronised calls update the "
                           "running statistics from the global batch inside the call; run the passes of a step in "
                           "order on one stream instead of deferring the updates")


class sync_batch_norm:
    """Context manager: synchronised BatchNorm over the ranks of ``process_group`` (default: the default group).

    Inside it, every training-mode ``bn_act`` call normalises with the statistics of the batches of all ranks together
    and updates the running statistics from them, as ``torch.nn.SyncBatchNorm`` does; its backward uses the global
    batch as well.  Each direction of a call runs a local phase, an all-gather of 3*C*V fp64 values per rank (rank
    order), and a global phase, so the ranks must issue the same BN calls in the same order.  With a world size of 1,
    and for eval-mode calls, nothing changes.  Not combinable with ``defer_bn_updates``."""

    def __init__(self, process_group: Optional["dist.ProcessGroup"] = None):
        self.group = process_group

    def __enter__(self):
        global _bn_sync
        sync = (self.group,)
        if _bn_defer is not None:
            _refuse_sync_with_defer(sync)
        self._prev, _bn_sync = _bn_sync, sync
        return self

    def __exit__(self, *exc):
        global _bn_sync
        _bn_sync = self._prev
        return False


def _all_gather_rows(rows, group):
    """[world * 3*C*V] fp64: every rank's rows in rank order (list form: NCCL and gloo both provide it)."""
    parts = [torch.empty_like(rows) for _ in range(dist.get_world_size(group))]
    dist.all_gather(parts, rows, group=group)
    return torch.cat(parts)


class _BnAct(torch.autograd.Function):

    @staticmethod
    def forward(ctx, y, r, gamma, beta, prelu, running_mean, running_var, nbt, mask, out_order, vc_order, training,
                eps, momentum, pass_r):
        sync = _bn_sync if training and _sync_world(_bn_sync) > 1 else None
        if sync is not None:
            if _bn_defer is not None:
                _refuse_sync_with_defer(sync)
            rows = _all_gather_rows(torch.ops.dstd_b200.bn_act_fwd_local(y, vc_order), sync[0])
            out, mean, invstd = torch.ops.dstd_b200.bn_act_fwd_global(y, r, gamma, beta, running_mean, running_var,
                                                                      nbt, prelu, mask, rows, out_order, vc_order,
                                                                      eps, momentum)
        else:
            deferred = _bn_defer is not None and training and running_mean is not None
            if deferred:
                n, _, t, _ = y.shape
                entry = [running_mean, running_var, nbt, float(momentum), float(eps), float(n * t)]
                running_mean = running_var = nbt = None
            out, mean, invstd = torch.ops.dstd_b200.bn_act_fwd(y, r, gamma, beta, running_mean, running_var, nbt,
                                                               prelu, mask, out_order, vc_order, training, eps,
                                                               momentum)
            if deferred:
                _bn_defer.append(entry + [mean, invstd])
        ctx.save_for_backward(y, r, gamma, beta, prelu, mask, mean, invstd)
        ctx.vc_order, ctx.training, ctx.pass_r = vc_order, training, pass_r
        ctx.sync = sync          # the backward performs its own exchange over the same group
        if pass_r:
            # second output = r itself: whatever else consumes r downstream (the layer skip) sends its gradient back
            # through this node, where the backward kernel adds it to d(pre-activation) in the same pass
            return out, r.view_as(r)
        return out

    @staticmethod
    def backward(ctx, gout, g_thru=None):
        y, r, gamma, beta, prelu, mask, mean, invstd = ctx.saved_tensors
        need_gr = r is not None and ctx.needs_input_grad[1]
        gr_add = g_thru if need_gr else None
        if ctx.sync is not None:
            gg, gb, gp, rows, gy, gr = torch.ops.dstd_b200.bn_act_bwd_local(y, r, gout, gamma, beta, prelu, mask,
                                                                            mean, invstd, ctx.vc_order, need_gr, gr_add)
            rows = _all_gather_rows(rows, ctx.sync[0])
            torch.ops.dstd_b200.bn_act_bwd_global(y, r, gout, gamma, beta, prelu, mask, mean, invstd, rows,
                                                  ctx.vc_order, gy, _opt(gr), gr_add)
        else:
            gy, gr, gg, gb, gp = torch.ops.dstd_b200.bn_act_bwd(y, r, gout, gamma, beta, prelu, mask, mean, invstd,
                                                                ctx.vc_order, ctx.training, need_gr, gr_add)
        return (gy, _opt(gr), gg, gb, _opt(gp), None, None, None, None, None, None, None, None, None, None)


def bn_act(y, bn: torch.nn.BatchNorm1d, r=None, prelu=None, mask=None, vc_order=False, out_order=ORDER_LIKE_INPUT,
           training=None, pass_r=False):
    """out = mask * prelu(BN(y) + r) on logical [N,C,T,V] tensors of any strides (BN over (N,T) per (c,v)).

    ``out_order``: memory order of the result (lets the op transpose T/V for free).
    ``pass_r``: also return ``r`` (as a second output of the same autograd node); use that alias for every other
    consumer of ``r`` and the gradients meet inside the BN backward kernel instead of in a separate add."""
    training = bn.training if training is None else training
    use_batch = training or bn.running_mean is None
    mom = 0.0 if bn.momentum is None else bn.momentum
    track = bn.track_running_stats and training
    return _BnAct.apply(y, r, bn.weight, bn.bias, prelu,
                        bn.running_mean if (track or not use_batch) else None,
                        bn.running_var if (track or not use_batch) else None,
                        bn.num_batches_tracked if track else None,
                        mask, out_order, vc_order, use_batch, bn.eps, mom, bool(pass_r and r is not None))


class _ChMix(torch.autograd.Function):

    @staticmethod
    def forward(ctx, x, w, b):
        ctx.save_for_backward(x, w)
        ctx.has_b = b is not None
        return torch.ops.dstd_b200.chmix_fwd(x, w, b)

    @staticmethod
    def backward(ctx, gout):
        x, w = ctx.saved_tensors
        gx, gw, gb = torch.ops.dstd_b200.chmix_bwd(x, gout, w, ctx.needs_input_grad[0])
        return _opt(gx), gw, (gb if ctx.has_b else None)


def chmix(xu, w, b=None):
    """1x1 channel mix on unit coordinates [N,C,P,K]."""
    return _ChMix.apply(xu, w, b)


class _Prep(torch.autograd.Function):

    @staticmethod
    def forward(ctx, x):
        return torch.ops.dstd_b200.prep_fwd(x)

    @staticmethod
    def backward(ctx, gh):
        return torch.ops.dstd_b200.prep_bwd(gh)


class _Finish(torch.autograd.Function):

    @staticmethod
    def forward(ctx, z, x):
        return torch.ops.dstd_b200.finish_fwd(z, x)

    @staticmethod
    def backward(ctx, gy):
        gz, gx = torch.ops.dstd_b200.finish_bwd(gy.contiguous(), ctx.needs_input_grad[1])
        return gz, _opt(gx)


def prep(x):
    """[N,T,V,3] -> motion-augmented [N,6,T,V] (model/dstdgcn.py:298-303)."""
    return _Prep.apply(x.contiguous())


def finish(z, x):
    """[N,3,T,V] (+ last observed frame of x) -> [N,T,V,3] (model/dstdgcn.py:314-315)."""
    return _Finish.apply(z, x.contiguous())


class _Mpjpe(torch.autograd.Function):
    """scale * mean ||pred - target||_2 ; the gradient is produced in the same kernel pass."""

    @staticmethod
    def forward(ctx, pred, target, scale):
        loss = torch.zeros((), dtype=torch.float32, device=pred.device)
        g = torch.ops.dstd_b200.mpjpe(pred, target, loss, scale, False)
        ctx.save_for_backward(g)
        return loss

    @staticmethod
    def backward(ctx, gl):
        (g,) = ctx.saved_tensors
        return g * gl, None, None


def mpjpe(pred, target, scale=1.0):
    """Mean per-joint position error (engine/utils/loss.py:52-65) with fused gradient."""
    return _Mpjpe.apply(pred.contiguous(), target.contiguous(), float(scale))
