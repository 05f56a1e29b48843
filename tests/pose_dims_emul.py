"""CPU emulation (fp64) of the head, tail and loss entry points of the C ABI for D coordinates per joint
(include/dstd_b200.h, ``dstd_{prep,finish}_{forward,backward}_d`` and ``dstd_pose_error_forward_backward``), with the
Python-level interface of ``dstd_gcn_b200._lib.CudaBackend``, so that a model of ``input_channels = 2 * D`` and
``TrainStep`` run on a CPU-only box.

It is a subclass kept with the tests rather than more methods of ``oracle/abi_emul.py``: ``oracle/`` is the pinned
reference the existing suite is checked against and stays unchanged.  The oracle's prep_forward, finish_forward and
finish_backward already take any D; prep_backward and the loss are restated here for any D."""
from __future__ import annotations

import torch

from oracle.abi_emul import EmulBackend


class PoseDimsEmulBackend(EmulBackend):
    """EmulBackend for x [N,T,V,D], any D."""

    name = "emul-dims"

    def prep_backward(self, gh):
        d = gh.shape[1] // 2
        g = gh.permute(0, 2, 3, 1)            # [N,T,V,2D]
        gx = (g[..., :d] + g[..., d:]).clone()
        gx[:, -1] -= g[..., d:].sum(dim=1)
        return gx.contiguous()

    def pose_error(self, pred, target, scale, loss_accum, accumulate, dims):
        loss_accum = loss_accum.view(())
        d = pred.reshape(-1, dims) - target.reshape(-1, dims)
        nrm = torch.sqrt((d * d).sum(dim=1))
        j = d.shape[0]
        loss = nrm.mean() * scale
        if accumulate:
            loss_accum += loss
        else:
            loss_accum.copy_(loss.reshape(loss_accum.shape))
        g = torch.where(nrm[:, None] > 0, d / nrm.clamp_min(1e-30)[:, None], torch.zeros_like(d)) * (scale / j)
        return g.reshape(pred.shape)
