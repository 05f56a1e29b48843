"""Batch construction of the reference datasets, done with device-side gathers (SURVEY.md 8f item 4).

The reference builds three views of every window on the host (dataset/h36m.py:53-63, same in cmu_mocap.py / pw3d.py)
and ships all of them over PCIe.  Here only the raw window ``all_seqs [N, T, 3J]`` has to reach the device; the model
input (observed frames + the last observed frame repeated), the time-reversed input used by the inverse pass and the
target are index gathers on the device."""
from typing import Optional, Sequence, Tuple

import torch


def window_indices(input_n: int, output_n: int, padding: bool = True) -> Tuple[torch.Tensor, torch.Tensor]:
    """Frame indices of the forward and the reversed input window (dataset/h36m.py:53-60).

    padding=True : forward  = [0 .. input_n-1] + output_n x [input_n-1]
                   reversed = [output_n+input_n-1 .. output_n] + output_n x [output_n]
    padding=False: forward  = [0 .. T-1], reversed = [T-1 .. 0]"""
    t = input_n + output_n
    if padding:
        fwd = torch.cat((torch.arange(0, input_n), torch.full((output_n,), input_n - 1)))
        inv = torch.cat((torch.arange(output_n + input_n - 1, output_n - 1, -1), torch.full((output_n,), output_n)))
    else:
        fwd = torch.arange(0, t)
        inv = torch.arange(t - 1, -1, -1)
    return fwd.long(), inv.long()


def window_batch(all_seqs: torch.Tensor, input_n: int, output_n: int, dim_used: Optional[Sequence[int]] = None,
                 padding: bool = True) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """``(inputs, inputs_inv, targets)`` of ``__getitem__`` (dataset/h36m.py:121-127) for a whole batch, on
    ``all_seqs``'s device.  ``all_seqs``: raw windows ``[N, input_n + output_n, 3J]``; ``dim_used``: coordinate columns
    the model sees (``None`` = all)."""
    assert all_seqs.dim() == 3 and all_seqs.shape[1] == input_n + output_n
    dev = all_seqs.device
    used = all_seqs if dim_used is None else all_seqs.index_select(
        2, torch.as_tensor(dim_used, dtype=torch.long, device=dev))
    fwd, inv = window_indices(input_n, output_n, padding)
    return used.index_select(1, fwd.to(dev)), used.index_select(1, inv.to(dev)), used


# joint groups swapped by the mirror augmentation (dataset/h36m.py:105-112)
_H36M_RIGHT = [1, 2, 3, 4, 5] + [16, 17, 18, 19, 20, 21, 22, 23]
_H36M_LEFT = [6, 7, 8, 9, 10] + [24, 25, 26, 27, 28, 29, 30, 31]


# (right, left) joint lists of the other datasets, verbatim from dataset/cmu.py:97-98 and dataset/pw3d.py:121-122.  The CMU
# lists are not a clean permutation (joint 24 is in both, 34 in neither): the reference's two assignments are
# reproduced in order, so the quirk is reproduced too.
_MIRROR = {
    "h36m": (_H36M_RIGHT, _H36M_LEFT),
    "cmu": ([2, 3, 4, 5, 6, 21, 22, 23, 24, 27, 25, 26, 28], [8, 9, 10, 11, 12, 30, 31, 32, 33, 36, 24, 35, 37]),
    "3dpw": ([1, 4, 7, 10, 13, 16, 18, 20, 22], [2, 5, 8, 11, 14, 17, 19, 21, 23]),
}


def _registered_mirror(layout: str):
    from .model.layers import graph
    lists = graph.mirror_lists(layout)      # KeyError for an unknown layout, as for the built-in table
    if lists is None:
        raise ValueError(f"layout {layout!r} was registered without mirror lists (register_layout(..., mirror=(right, left)))")
    return lists


def mirror(all_seqs: torch.Tensor, layout: str, dims: int = 3) -> torch.Tensor:
    """Left/right mirrored copy of raw windows ``[N, T, D*J]`` of ``dims`` = D coordinates per joint (``get_mirror`` of
    dataset/h36m.py:100-116, dataset/cmu.py:93-105, dataset/pw3d.py:116-128): `m[right] = src[left]`, then
    `m[left] = src[right]`, then negate coordinate 0 (x).  Runs on the tensor's device.  A layout added with
    ``graph.register_layout`` uses the lists registered with it."""
    right, left = _MIRROR[layout] if layout in _MIRROR else _registered_mirror(layout)
    n, t, vc = all_seqs.shape
    src = all_seqs.view(n, t, vc // dims, dims)
    dev = all_seqs.device
    r, l = torch.as_tensor(right, device=dev), torch.as_tensor(left, device=dev)
    out = src.clone()
    out[:, :, r] = src[:, :, l]
    out[:, :, l] = src[:, :, r]
    out[..., 0] = -out[..., 0]
    return out.view(n, t, vc)


def mirror_h36m(all_seqs: torch.Tensor) -> torch.Tensor:
    return mirror(all_seqs, "h36m")


class DevicePrefetcher:
    """Pinned, double-buffered host->device feed of raw windows (SURVEY.md 8f item 4).

    The reference uploads three tensors per step with ``.cuda(non_blocking=True)`` from a pinned DataLoader
    (runner/h36m.py:35-54, engine/prediction.py:223-225).  Here only ``all_seqs`` crosses PCIe: batch i+1 is copied
    from a pinned staging buffer on a side stream while batch i trains, and ``(inputs, inputs_inv, targets)`` are
    device-side gathers of it (``window_batch``), optionally with the mirrored copy appended (``mirror``).

        for inputs, inputs_inv, targets, all_seqs in DevicePrefetcher(loader, 10, 25, dim_used, device="cuda"): ...

    ``batches`` yields CPU tensors / arrays ``[N, T, D*J]`` (or tuples whose LAST element is that, like the reference's
    dataset tuple); ``dims`` = D coordinates per joint is what ``mirror`` needs."""

    def __init__(self, batches, input_n, output_n, dim_used=None, padding=True, device="cuda", mirror_layout=None,
                 depth=2, dims=3):
        self.batches, self.input_n, self.output_n = batches, input_n, output_n
        self.dim_used, self.padding, self.mirror_layout, self.dims = dim_used, padding, mirror_layout, dims
        self.device = torch.device(device)
        self.depth = max(1, int(depth))
        self.cuda = self.device.type == "cuda"
        self.stream = torch.cuda.Stream(self.device) if self.cuda else None
        self._pinned = [None] * self.depth

    def _stage(self, slot, raw):
        raw = raw[-1] if isinstance(raw, (tuple, list)) else raw
        raw = torch.as_tensor(raw).float()
        if not self.cuda:
            return raw, None
        buf = self._pinned[slot]
        if buf is None or buf.shape != raw.shape:
            buf = self._pinned[slot] = torch.empty(raw.shape, dtype=torch.float32).pin_memory()
        buf.copy_(raw)
        with torch.cuda.stream(self.stream):
            dev = buf.to(self.device, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.stream)
        return dev, ev

    def __iter__(self):
        it = iter(self.batches)
        queue = []
        slot = 0
        for raw in it:
            queue.append(self._stage(slot, raw))
            slot = (slot + 1) % self.depth
            if len(queue) >= self.depth:
                yield self._finish(*queue.pop(0))
        while queue:
            yield self._finish(*queue.pop(0))

    def _finish(self, dev, ev):
        if ev is not None:
            torch.cuda.current_stream(self.device).wait_event(ev)
            dev.record_stream(torch.cuda.current_stream(self.device))
        if self.mirror_layout is not None:
            dev = torch.cat((dev, mirror(dev, self.mirror_layout, self.dims)), dim=0)
        a, b, c = window_batch(dev, self.input_n, self.output_n, self.dim_used, self.padding)
        return a, b, c, dev
