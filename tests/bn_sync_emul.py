"""CPU emulation (fp64) of the synchronised-BatchNorm entry points of the C ABI (include/dstd_b200.h,
``dstd_bn_act_{forward,backward}_{local,global}``), on top of the ABI emulation in ``oracle/abi_emul.py``: the same
Python-level interface as ``dstd_gcn_b200._lib.CudaBackend``, so the whole synchronised wiring (ops, autograd,
``TrainStep(sync_bn=True)`` over gloo) runs on a CPU-only box.

It is a subclass kept with the tests rather than four more methods of ``oracle/abi_emul.py``: ``oracle/`` is the
pinned reference the existing suite is checked against and stays unchanged; the subclass only adds the split phases
and reuses the oracle's plain BatchNorm emulation for everything they share."""
from __future__ import annotations

import torch

from oracle.abi_emul import EmulBackend


class SyncEmulBackend(EmulBackend):
    """EmulBackend plus the four phases of synchronised BatchNorm.  Exchange rows: fp64 [3][C*V] per rank in BN
    parameter order, (count, mean, M2) in the forward and (count, sum g', sum g' xhat) in the backward."""

    name = "emul-sync"

    @staticmethod
    def _rows(all_rows, c, v):
        return all_rows.double().view(-1, 3, c * v)                  # [world, 3, C*V]

    def bn_act_forward_local(self, y, vc_order):
        n, c, t, v = y.shape
        yd = y.double()
        mean = yd.mean(dim=(0, 2))
        m2 = ((yd - mean.view(1, c, 1, v)) ** 2).sum(dim=(0, 2))
        cnt = torch.full((c * v,), float(n * t), dtype=torch.float64)
        return torch.cat((cnt, self._bn_unindex(mean, vc_order), self._bn_unindex(m2, vc_order)))

    def bn_act_forward_global(self, y, r, gamma, beta, running_mean, running_var, nbt, prelu, mask, vc_order, eps,
                              momentum, all_rows, out_like=None):
        n, c, t, v = y.shape
        rows = self._rows(all_rows, c, v)
        cnt = rows[:, 0].sum(dim=0)
        mean = (rows[:, 0] * rows[:, 1]).sum(dim=0) / cnt
        m2 = (rows[:, 2] + rows[:, 0] * (rows[:, 1] - mean) ** 2).sum(dim=0)
        var = m2 / cnt
        if running_mean is not None:
            unb = m2 / (cnt - 1).clamp_min(1)
            running_mean.mul_(1 - momentum).add_(momentum * mean.to(running_mean.dtype))
            running_var.mul_(1 - momentum).add_(momentum * unb.to(running_var.dtype))
        if nbt is not None:
            nbt += 1
        # the eval branch of the plain call normalises with the statistics it is given
        return self.bn_act_forward(y, r, gamma, beta, mean.to(y.dtype), var.to(y.dtype), None, prelu, mask, vc_order,
                                   False, eps, momentum, out_like)

    def _gpre_xhat(self, y, r, gout, gamma, beta, prelu, mask, save_mean, save_invstd, vc_order):
        n, c, t, v = y.shape
        mean = self._bn_index(save_mean, c, v, vc_order)
        invstd = self._bn_index(save_invstd, c, v, vc_order)
        g_, b_ = self._bn_index(gamma, c, v, vc_order), self._bn_index(beta, c, v, vc_order)
        xhat = (y - mean) * invstd
        ga = gout * mask.view(n, c, t, v) if mask is not None else gout
        if prelu is not None:
            pre = xhat * g_ + b_
            if r is not None:
                pre = pre + r
            ga = ga * torch.where(pre > 0, torch.ones_like(pre), prelu.reshape(()).expand_as(pre))
        return ga, xhat, g_ * invstd

    def bn_act_backward_local(self, y, r, gout, gamma, beta, prelu, mask, save_mean, save_invstd, vc_order,
                              need_gr=True, gr_add=None):
        n, c, t, v = y.shape
        _, _, ggamma, gbeta, gprelu = self.bn_act_backward(y, r, gout, gamma, beta, prelu, mask, save_mean,
                                                           save_invstd, vc_order, False, need_gr, gr_add)
        cnt = torch.full((c * v,), float(n * t), dtype=torch.float64)
        gy = torch.empty_like(y)
        gr = torch.empty_like(r) if (r is not None and need_gr) else None
        return ggamma, gbeta, gprelu, torch.cat((cnt, gbeta.double(), ggamma.double())), gy, gr

    def bn_act_backward_global(self, y, r, gout, gamma, beta, prelu, mask, save_mean, save_invstd, vc_order, all_rows,
                               gy, gr=None, gr_add=None):
        n, c, t, v = y.shape
        rows = self._rows(all_rows, c, v)
        cnt = rows[:, 0].sum(dim=0)
        k1 = self._bn_index((rows[:, 1].sum(dim=0) / cnt).to(y.dtype), c, v, vc_order)
        k2 = self._bn_index((rows[:, 2].sum(dim=0) / cnt).to(y.dtype), c, v, vc_order)
        gpre, xhat, gi = self._gpre_xhat(y, r, gout, gamma, beta, prelu, mask, save_mean, save_invstd, vc_order)
        gy.copy_(gi * (gpre - k1 - xhat * k2))
        if gr is not None:
            gr.copy_(gpre if gr_add is None else gpre + gr_add)
        return gy, gr
