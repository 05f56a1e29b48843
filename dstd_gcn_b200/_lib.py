"""ctypes binding of ``libdstd_b200.so`` (C ABI in ``include/dstd_b200.h``) and the CUDA backend.

There is deliberately no CPU implementation here: if the shared library is
missing, or a tensor is not a CUDA fp32 tensor, the call raises.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DSTD_B200_LIB") or os.path.join(_HERE, "csrc", "libdstd_b200.so")   # override: A/B builds

MAX_BRANCH = 2
FLAG_ADJ_T = 1

_f32p = C.POINTER(C.c_float)


class View(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("sn", C.c_longlong), ("sc", C.c_longlong), ("sp", C.c_longlong),
                ("sk", C.c_longlong)]


class Branch(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in
                ("w_m1", "b_m1", "w_m2", "b_m2", "w_rm", "b_rm", "w_f", "b_f", "adj", "adj_w", "adj_r")]


class BranchGrad(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in
                ("w_m1", "b_m1", "w_m2", "b_m2", "w_rm", "b_rm", "w_f", "b_f", "adj_eff", "adj_w")]


class GcFwdArgs(C.Structure):
    _fields_ = [("N", C.c_int), ("Cin", C.c_int), ("Cout", C.c_int), ("P", C.c_int), ("K", C.c_int),
                ("nb", C.c_int), ("flags", C.c_int),
                ("x", View), ("out", View), ("skip", View), ("alpha", C.c_void_p),
                ("br", Branch * MAX_BRANCH),
                ("m", C.c_void_p), ("pd", C.c_void_p), ("xa", C.c_void_p),
                ("ws", C.c_void_p), ("ws_bytes", C.c_size_t)]


class GcBwdArgs(C.Structure):
    _fields_ = [("N", C.c_int), ("Cin", C.c_int), ("Cout", C.c_int), ("P", C.c_int), ("K", C.c_int),
                ("nb", C.c_int), ("flags", C.c_int),
                ("x", View), ("gout", View), ("gx", View), ("alpha", C.c_void_p),
                ("br", Branch * MAX_BRANCH),
                ("m", C.c_void_p), ("pd", C.c_void_p), ("xa", C.c_void_p),
                ("gbr", BranchGrad * MAX_BRANCH), ("galpha", C.c_void_p),
                ("ws", C.c_void_p), ("ws_bytes", C.c_size_t), ("gx_add", View)]


class BnFwdArgs(C.Structure):
    _fields_ = [("N", C.c_int), ("C", C.c_int), ("T", C.c_int), ("V", C.c_int),
                ("vc_order", C.c_int), ("training", C.c_int), ("eps", C.c_float), ("momentum", C.c_float),
                ("y", View), ("r", View), ("out", View),
                ("gamma", C.c_void_p), ("beta", C.c_void_p),
                ("running_mean", C.c_void_p), ("running_var", C.c_void_p), ("num_batches_tracked", C.c_void_p),
                ("prelu", C.c_void_p), ("mask", C.c_void_p),
                ("save_mean", C.c_void_p), ("save_invstd", C.c_void_p),
                ("ws", C.c_void_p), ("ws_bytes", C.c_size_t)]


class BnBwdArgs(C.Structure):
    _fields_ = [("N", C.c_int), ("C", C.c_int), ("T", C.c_int), ("V", C.c_int),
                ("vc_order", C.c_int), ("training", C.c_int),
                ("y", View), ("r", View), ("gout", View), ("gy", View), ("gr", View),
                ("gamma", C.c_void_p), ("beta", C.c_void_p), ("prelu", C.c_void_p), ("mask", C.c_void_p),
                ("save_mean", C.c_void_p), ("save_invstd", C.c_void_p),
                ("ggamma", C.c_void_p), ("gbeta", C.c_void_p), ("gprelu", C.c_void_p),
                ("ws", C.c_void_p), ("ws_bytes", C.c_size_t), ("gr_add", View)]


class ChmixFwdArgs(C.Structure):
    _fields_ = [("N", C.c_int), ("Cin", C.c_int), ("Cout", C.c_int), ("P", C.c_int), ("K", C.c_int),
                ("x", View), ("out", View), ("w", C.c_void_p), ("b", C.c_void_p)]


class ChmixBwdArgs(C.Structure):
    _fields_ = [("N", C.c_int), ("Cin", C.c_int), ("Cout", C.c_int), ("P", C.c_int), ("K", C.c_int),
                ("x", View), ("gout", View), ("gx", View), ("w", C.c_void_p),
                ("gw", C.c_void_p), ("gb", C.c_void_p), ("ws", C.c_void_p), ("ws_bytes", C.c_size_t)]


# every symbol include/dstd_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "dstd_gc_needs_xa": (C.c_int, [C.c_int] * 5),
    "dstd_gc_fwd_workspace_bytes": (C.c_size_t, [C.c_int] * 6),
    "dstd_gc_bwd_workspace_bytes": (C.c_size_t, [C.c_int] * 6),
    "dstd_gc_forward": (C.c_int, [C.POINTER(GcFwdArgs), C.c_void_p]),
    "dstd_gc_backward": (C.c_int, [C.POINTER(GcBwdArgs), C.c_void_p]),
    "dstd_bn_act_workspace_bytes": (C.c_size_t, [C.c_int] * 4),
    "dstd_bn_act_forward": (C.c_int, [C.POINTER(BnFwdArgs), C.c_void_p]),
    "dstd_bn_act_backward": (C.c_int, [C.POINTER(BnBwdArgs), C.c_void_p]),
    "dstd_bn_sync_buffer_doubles": (C.c_size_t, [C.c_int, C.c_int]),
    "dstd_bn_act_forward_local": (C.c_int, [C.POINTER(BnFwdArgs), C.c_void_p, C.c_void_p]),
    "dstd_bn_act_forward_global": (C.c_int, [C.POINTER(BnFwdArgs), C.c_void_p, C.c_int, C.c_void_p]),
    "dstd_bn_act_backward_local": (C.c_int, [C.POINTER(BnBwdArgs), C.c_void_p, C.c_void_p]),
    "dstd_bn_act_backward_global": (C.c_int, [C.POINTER(BnBwdArgs), C.c_void_p, C.c_int, C.c_void_p]),
    "dstd_chmix_bwd_workspace_bytes": (C.c_size_t, [C.c_int] * 5),
    "dstd_chmix_forward": (C.c_int, [C.POINTER(ChmixFwdArgs), C.c_void_p]),
    "dstd_chmix_backward": (C.c_int, [C.POINTER(ChmixBwdArgs), C.c_void_p]),
    "dstd_prep_forward": (C.c_int, [C.c_void_p, View, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "dstd_prep_backward": (C.c_int, [View, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "dstd_finish_forward": (C.c_int, [View, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "dstd_finish_backward": (C.c_int, [C.c_void_p, View, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "dstd_mpjpe_workspace_bytes": (C.c_size_t, [C.c_longlong]),
    "dstd_mpjpe_forward_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_float, C.c_int, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dstd_adam_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_float, C.c_float,
                                 C.c_float, C.c_float, C.c_float, C.c_float, C.c_int, C.c_void_p, C.c_void_p,
                                 C.c_void_p]),
    "dstd_last_error": (C.c_char_p, []),
    "dstd_version": (C.c_char_p, []),
    "dstd_kernel_launch_count": (C.c_int, []),
    "dstd_device_error": (C.c_int, [C.c_int]),
    "dstd_debug_raise_device_error": (C.c_int, [C.c_int, C.c_void_p]),
}

_lib = None


def load_library(path: str = LIB_PATH):
    """dlopen the C-ABI library and type every exported symbol.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(path):
        raise RuntimeError(
            f"dstd_gcn_b200: CUDA library not built ({path}). Run `python -c 'import __graft_entry__ as g; "
            "g.build()'` (nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)       # AttributeError => header/library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _check(t, what, dtype=torch.float32):
    if t is None:
        return
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"dstd_gcn_b200: `{what}` must be a CUDA tensor (the hot path has no CPU fallback)")
    if t.dtype != dtype:
        raise RuntimeError(f"dstd_gcn_b200: `{what}` must be {dtype}, got {t.dtype}")
    if t.device.index is not None and t.device.index != torch.cuda.current_device():
        # the library launches on the CURRENT device (it never switches devices); a tensor elsewhere would be an
        # illegal access.  One process per GPU is the supported layout: torch.cuda.set_device(local_rank) first.
        raise RuntimeError(f"dstd_gcn_b200: `{what}` lives on cuda:{t.device.index} but the current device is "
                           f"cuda:{torch.cuda.current_device()} (call torch.cuda.set_device first)")


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _cptr(t, what):
    """Pointer of a tensor that the ABI reads as a dense array."""
    if t is None:
        return None
    _check(t, what)
    if not t.is_contiguous():
        raise RuntimeError(f"dstd_gcn_b200: `{what}` must be contiguous")
    return C.c_void_p(t.data_ptr())


def _view(t, what):
    if t is None:
        return View(None, 0, 0, 0, 0)
    _check(t, what)
    assert t.dim() == 4, what
    s = t.stride()
    return View(C.c_void_p(t.data_ptr()), s[0], s[1], s[2], s[3])


def _like_layout(ref, channels):
    shape = list(ref.shape)
    shape[1] = channels
    order = sorted(range(ref.dim()), key=lambda d: (ref.stride(d), ref.shape[d]), reverse=True)
    strides = [0] * ref.dim()
    acc = 1
    for d in reversed(order):
        strides[d] = acc
        acc *= shape[d]
    return torch.empty_strided(shape, strides, dtype=ref.dtype, device=ref.device)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


_BR_KEYS = ("w_m1", "b_m1", "w_m2", "b_m2", "w_rm", "b_rm", "w_f", "b_f", "adj", "adj_w", "adj_r")
_GR_KEYS = ("w_m1", "b_m1", "w_m2", "b_m2", "w_rm", "b_rm", "w_f", "b_f")


class CudaBackend:
    """Tensor-level wrapper: allocates outputs/workspaces with torch, fills the arg structs, calls the C ABI."""

    name = "cuda"

    def __init__(self):
        self.lib = load_library()

    # -- helpers
    def _ok(self, rc, fn):
        if rc != 0:
            msg = self.lib.dstd_last_error()
            raise RuntimeError(f"{fn} failed ({rc}): {msg.decode() if msg else ''}")

    @property
    def launches(self):
        return int(self.lib.dstd_kernel_launch_count())

    @staticmethod
    def _ws(nbytes, device):
        return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)

    def _fill_branches(self, arr, brs):
        for i, br in enumerate(brs):
            for k in _BR_KEYS:
                setattr(arr[i], k, _cptr(br.get(k), k))

    # -- DSTD-GC unit
    def gc_forward(self, xu, alpha, brs, skip_u, adj_t):
        n, cin, p_, k_ = xu.shape
        nb = len(brs)
        cout = brs[0]["w_f"].shape[0]
        dev = xu.device
        out = _like_layout(xu, cout)
        m = torch.empty((n, nb, 4, p_, k_), dtype=torch.float32, device=dev)
        pd = torch.empty((n, nb, p_, k_, k_), dtype=torch.float32, device=dev)
        # the aggregated tile is only kept for shapes whose backward cannot recompute it on chip
        need_xa = bool(self.lib.dstd_gc_needs_xa(cin, cout, p_, k_, nb))
        xa = torch.empty((n, nb, cin + 1, p_, k_) if need_xa else (0,), dtype=torch.float32, device=dev)
        ws = self._ws(self.lib.dstd_gc_fwd_workspace_bytes(n, cin, cout, p_, k_, nb), dev)
        a = GcFwdArgs()
        a.N, a.Cin, a.Cout, a.P, a.K, a.nb = n, cin, cout, p_, k_, nb
        a.flags = FLAG_ADJ_T if adj_t else 0
        a.x, a.out, a.skip = _view(xu, "x"), _view(out, "out"), _view(skip_u, "skip")
        a.alpha = _cptr(alpha, "alpha")
        self._fill_branches(a.br, brs)
        a.m, a.pd, a.xa = _ptr(m), _ptr(pd), (_ptr(xa) if xa.numel() else None)
        a.ws, a.ws_bytes = _ptr(ws), ws.numel()
        self._ok(self.lib.dstd_gc_forward(C.byref(a), _stream()), "dstd_gc_forward")
        return out, m, pd, xa

    def gc_backward(self, xu, gout_u, alpha, brs, m, pd, xa, adj_t, need_galpha=True, gx_add=None):
        n, cin, p_, k_ = xu.shape
        nb = len(brs)
        cout = brs[0]["w_f"].shape[0]
        dev = xu.device
        gx = torch.empty_like(xu)
        galpha = torch.empty((1,), dtype=torch.float32, device=dev) if alpha is not None else None
        ws = self._ws(self.lib.dstd_gc_bwd_workspace_bytes(n, cin, cout, p_, k_, nb), dev)
        a = GcBwdArgs()
        a.N, a.Cin, a.Cout, a.P, a.K, a.nb = n, cin, cout, p_, k_, nb
        a.flags = FLAG_ADJ_T if adj_t else 0
        a.x, a.gout, a.gx = _view(xu, "x"), _view(gout_u, "gout"), _view(gx, "gx")
        a.gx_add = _view(gx_add, "gx_add")
        a.alpha = _cptr(alpha, "alpha")
        self._fill_branches(a.br, brs)
        a.m, a.pd, a.xa = _cptr(m, "m"), _cptr(pd, "pd"), (_cptr(xa, "xa") if xa is not None and xa.numel() else None)
        grads = []
        for i, br in enumerate(brs):
            g = {k: torch.empty_like(br[k]) for k in _GR_KEYS}
            g["adj_eff"] = torch.empty((k_, k_), dtype=torch.float32, device=dev)
            g["adj_w"] = torch.empty((k_, k_), dtype=torch.float32, device=dev) if br.get("adj_w") is not None else None
            for k in _GR_KEYS + ("adj_eff", "adj_w"):
                setattr(a.gbr[i], k, _ptr(g[k]))
            grads.append(g)
        a.galpha = _ptr(galpha)
        a.ws, a.ws_bytes = _ptr(ws), ws.numel()
        self._ok(self.lib.dstd_gc_backward(C.byref(a), _stream()), "dstd_gc_backward")
        return gx, galpha, grads

    # -- BN + residual + PReLU + mask
    def _bn_fwd_args(self, y, r, gamma, beta, running_mean, running_var, nbt, prelu, mask, vc_order, training, eps,
                     momentum, out_like, with_ws=True):
        """Fills dstd_bn_act_fwd_args; returns (args, out, save_mean, save_invstd, workspace or None)."""
        n, c, t, v = y.shape
        dev = y.device
        out = torch.empty_like(out_like if out_like is not None else y, device=dev)
        save_mean = torch.empty((c * v,), dtype=torch.float32, device=dev)
        save_invstd = torch.empty((c * v,), dtype=torch.float32, device=dev)
        ws = self._ws(self.lib.dstd_bn_act_workspace_bytes(n, c, t, v), dev) if with_ws else None
        if nbt is not None:
            _check(nbt, "num_batches_tracked", torch.int64)
        a = BnFwdArgs()
        a.N, a.C, a.T, a.V = n, c, t, v
        a.vc_order, a.training, a.eps, a.momentum = int(vc_order), int(training), eps, momentum
        a.y, a.r, a.out = _view(y, "y"), _view(r, "r"), _view(out, "out")
        a.gamma, a.beta = _cptr(gamma, "gamma"), _cptr(beta, "beta")
        a.running_mean, a.running_var = _cptr(running_mean, "running_mean"), _cptr(running_var, "running_var")
        a.num_batches_tracked = _ptr(nbt)
        a.prelu, a.mask = _cptr(prelu, "prelu"), _cptr(mask, "mask")
        a.save_mean, a.save_invstd = _ptr(save_mean), _ptr(save_invstd)
        a.ws, a.ws_bytes = _ptr(ws), (ws.numel() if ws is not None else 0)
        return a, out, save_mean, save_invstd, ws

    def bn_act_forward(self, y, r, gamma, beta, running_mean, running_var, nbt, prelu, mask, vc_order, training,
                       eps, momentum, out_like=None):
        a, out, save_mean, save_invstd, ws = self._bn_fwd_args(y, r, gamma, beta, running_mean, running_var, nbt, prelu,
                                                               mask, vc_order, training, eps, momentum, out_like)
        self._ok(self.lib.dstd_bn_act_forward(C.byref(a), _stream()), "dstd_bn_act_forward")
        return out, save_mean, save_invstd

    @staticmethod
    def _bn_grad_bufs(y, r, prelu, need_gr):
        """gy, gr (None unless r and need_gr), ggamma, gbeta, gprelu (None without PReLU): uninitialised."""
        n, c, t, v = y.shape
        dev = y.device
        gr = torch.empty_like(r) if (r is not None and need_gr) else None
        gprelu = torch.empty((1,), dtype=torch.float32, device=dev) if prelu is not None else None
        return (torch.empty_like(y), gr, torch.empty((c * v,), dtype=torch.float32, device=dev),
                torch.empty((c * v,), dtype=torch.float32, device=dev), gprelu)

    def _bn_bwd_args(self, y, r, gout, gamma, beta, prelu, mask, save_mean, save_invstd, vc_order, training, gy, gr,
                     gr_add, ggamma=None, gbeta=None, gprelu=None, ws=None):
        """Fills dstd_bn_act_bwd_args with the given output buffers (None = not passed)."""
        n, c, t, v = y.shape
        a = BnBwdArgs()
        a.N, a.C, a.T, a.V = n, c, t, v
        a.vc_order, a.training = int(vc_order), int(training)
        a.y, a.r, a.gout = _view(y, "y"), _view(r, "r"), _view(gout, "gout")
        a.gy, a.gr = _view(gy, "gy"), _view(gr, "gr")
        a.gr_add = _view(gr_add if gr is not None else None, "gr_add")
        a.gamma, a.beta = _cptr(gamma, "gamma"), _cptr(beta, "beta")
        a.prelu, a.mask = _cptr(prelu, "prelu"), _cptr(mask, "mask")
        a.save_mean, a.save_invstd = _cptr(save_mean, "save_mean"), _cptr(save_invstd, "save_invstd")
        a.ggamma, a.gbeta, a.gprelu = _ptr(ggamma), _ptr(gbeta), _ptr(gprelu)
        a.ws, a.ws_bytes = _ptr(ws), (ws.numel() if ws is not None else 0)
        return a

    def bn_act_backward(self, y, r, gout, gamma, beta, prelu, mask, save_mean, save_invstd, vc_order, training,
                        need_gr=True, gr_add=None):
        n, c, t, v = y.shape
        gy, gr, ggamma, gbeta, gprelu = self._bn_grad_bufs(y, r, prelu, need_gr)
        ws = self._ws(self.lib.dstd_bn_act_workspace_bytes(n, c, t, v), y.device)
        a = self._bn_bwd_args(y, r, gout, gamma, beta, prelu, mask, save_mean, save_invstd, vc_order, training, gy, gr,
                              gr_add, ggamma, gbeta, gprelu, ws)
        self._ok(self.lib.dstd_bn_act_backward(C.byref(a), _stream()), "dstd_bn_act_backward")
        return gy, gr, ggamma, gbeta, gprelu

    # -- synchronised BN: the two phases of each direction around an all-gather of fp64 rows (include/dstd_b200.h)
    def _bn_rows(self, y, rows, what):
        n, c, t, v = y.shape
        _check(rows, what, torch.float64)
        per = int(self.lib.dstd_bn_sync_buffer_doubles(c, v))
        if not rows.is_contiguous() or rows.numel() % per:
            raise RuntimeError(f"dstd_gcn_b200: `{what}` must be a contiguous multiple of {per} doubles")
        return rows.numel() // per

    def bn_act_forward_local(self, y, vc_order):
        """This rank's exchange rows (count, mean, M2) [3*C*V] fp64 of a training-mode BN over y."""
        n, c, t, v = y.shape
        rows = torch.empty((int(self.lib.dstd_bn_sync_buffer_doubles(c, v)),), dtype=torch.float64, device=y.device)
        ws = self._ws(self.lib.dstd_bn_act_workspace_bytes(n, c, t, v), y.device)
        a = BnFwdArgs()
        a.N, a.C, a.T, a.V = n, c, t, v
        a.vc_order, a.training = int(vc_order), 1
        a.y = _view(y, "y")
        a.ws, a.ws_bytes = _ptr(ws), ws.numel()
        self._ok(self.lib.dstd_bn_act_forward_local(C.byref(a), _ptr(rows), _stream()), "dstd_bn_act_forward_local")
        return rows

    def bn_act_forward_global(self, y, r, gamma, beta, running_mean, running_var, nbt, prelu, mask, vc_order, eps,
                              momentum, all_rows, out_like=None):
        """Statistics merged from the gathered rows of every rank; same results as bn_act_forward."""
        world = self._bn_rows(y, all_rows, "all_rows")
        a, out, save_mean, save_invstd, _ = self._bn_fwd_args(y, r, gamma, beta, running_mean, running_var, nbt, prelu,
                                                              mask, vc_order, True, eps, momentum, out_like,
                                                              with_ws=False)
        self._ok(self.lib.dstd_bn_act_forward_global(C.byref(a), _ptr(all_rows), world, _stream()),
                 "dstd_bn_act_forward_global")
        return out, save_mean, save_invstd

    def bn_act_backward_local(self, y, r, gout, gamma, beta, prelu, mask, save_mean, save_invstd, vc_order,
                              need_gr=True, gr_add=None):
        """This rank's parameter gradients and exchange rows (count, sum g', sum g' xhat) [3*C*V] fp64, plus the
        (not yet written) gy / gr buffers for bn_act_backward_global: their layouts pick the kernels of both phases."""
        n, c, t, v = y.shape
        gy, gr, ggamma, gbeta, gprelu = self._bn_grad_bufs(y, r, prelu, need_gr)
        ws = self._ws(self.lib.dstd_bn_act_workspace_bytes(n, c, t, v), y.device)
        a = self._bn_bwd_args(y, r, gout, gamma, beta, prelu, mask, save_mean, save_invstd, vc_order, True, gy, gr,
                              gr_add, ggamma, gbeta, gprelu, ws)
        rows = torch.empty((int(self.lib.dstd_bn_sync_buffer_doubles(c, v)),), dtype=torch.float64, device=y.device)
        self._ok(self.lib.dstd_bn_act_backward_local(C.byref(a), _ptr(rows), _stream()), "dstd_bn_act_backward_local")
        return ggamma, gbeta, gprelu, rows, gy, gr

    def bn_act_backward_global(self, y, r, gout, gamma, beta, prelu, mask, save_mean, save_invstd, vc_order, all_rows,
                               gy, gr=None, gr_add=None):
        """Writes gy (and gr) of the global batch, from the gathered rows of every rank, into the buffers that
        bn_act_backward_local returned; returns them."""
        world = self._bn_rows(y, all_rows, "all_rows")
        a = self._bn_bwd_args(y, r, gout, gamma, beta, prelu, mask, save_mean, save_invstd, vc_order, True, gy, gr,
                              gr_add)
        self._ok(self.lib.dstd_bn_act_backward_global(C.byref(a), _ptr(all_rows), world, _stream()),
                 "dstd_bn_act_backward_global")
        return gy, gr

    # -- 1x1 channel mix
    def chmix_forward(self, xu, w, b):
        n, cin, p_, k_ = xu.shape
        cout = w.shape[0]
        out = _like_layout(xu, cout)
        a = ChmixFwdArgs()
        a.N, a.Cin, a.Cout, a.P, a.K = n, cin, cout, p_, k_
        a.x, a.out = _view(xu, "x"), _view(out, "out")
        a.w, a.b = _cptr(w, "w"), _cptr(b, "b")
        self._ok(self.lib.dstd_chmix_forward(C.byref(a), _stream()), "dstd_chmix_forward")
        return out

    def chmix_backward(self, xu, gout, w, need_gx=True):
        n, cin, p_, k_ = xu.shape
        cout = w.shape[0]
        dev = xu.device
        gx = torch.empty_like(xu) if need_gx else None
        gw = torch.empty_like(w)
        gb = torch.empty((cout,), dtype=torch.float32, device=dev)
        ws = self._ws(self.lib.dstd_chmix_bwd_workspace_bytes(n, cin, cout, p_, k_), dev)
        a = ChmixBwdArgs()
        a.N, a.Cin, a.Cout, a.P, a.K = n, cin, cout, p_, k_
        a.x, a.gout, a.gx = _view(xu, "x"), _view(gout, "gout"), _view(gx, "gx")
        a.w, a.gw, a.gb = _cptr(w, "w"), _ptr(gw), _ptr(gb)
        a.ws, a.ws_bytes = _ptr(ws), ws.numel()
        self._ok(self.lib.dstd_chmix_backward(C.byref(a), _stream()), "dstd_chmix_backward")
        return gx, gw, gb

    # -- head / tail
    def prep_forward(self, x):
        n, t, v, c = x.shape
        assert c == 3
        h = torch.empty((n, 6, t, v), dtype=torch.float32, device=x.device)
        self._ok(self.lib.dstd_prep_forward(_cptr(x, "x"), _view(h, "h"), n, t, v, _stream()), "dstd_prep_forward")
        return h

    def prep_backward(self, gh):
        n, _, t, v = gh.shape
        gx = torch.empty((n, t, v, 3), dtype=torch.float32, device=gh.device)
        self._ok(self.lib.dstd_prep_backward(_view(gh, "gh"), _ptr(gx), n, t, v, _stream()), "dstd_prep_backward")
        return gx

    def finish_forward(self, z, x):
        n, t, v, _ = x.shape
        y = torch.empty_like(x)
        self._ok(self.lib.dstd_finish_forward(_view(z, "z"), _cptr(x, "x"), _ptr(y), n, t, v, _stream()),
                 "dstd_finish_forward")
        return y

    def finish_backward(self, gy, need_gx=True):
        n, t, v, _ = gy.shape
        gz = torch.empty((n, 3, t, v), dtype=torch.float32, device=gy.device)
        gx = torch.empty_like(gy) if need_gx else None
        self._ok(self.lib.dstd_finish_backward(_cptr(gy, "gy"), _view(gz, "gz"), _ptr(gx), n, t, v, _stream()),
                 "dstd_finish_backward")
        return gz, gx

    # -- engine glue
    def mpjpe(self, pred, target, scale, loss_accum, accumulate):
        j = pred.numel() // 3
        gpred = torch.empty_like(pred)
        ws = self._ws(self.lib.dstd_mpjpe_workspace_bytes(j), pred.device)
        self._ok(self.lib.dstd_mpjpe_forward_backward(_cptr(pred, "pred"), _cptr(target, "target"), j, scale,
                                                      int(accumulate), _cptr(loss_accum, "loss"), _ptr(gpred),
                                                      _ptr(ws), ws.numel(), _stream()), "dstd_mpjpe_forward_backward")
        return gpred

    def adam_step(self, param, grad, exp_avg, exp_avg_sq, lr, beta1, beta2, eps, weight_decay, grad_scale, step,
                  lr_dev=None, step_dev=None):
        if lr_dev is not None:
            _check(lr_dev, "lr_dev")
        if step_dev is not None:
            _check(step_dev, "step_dev", torch.int32)
        self._ok(self.lib.dstd_adam_step(_cptr(param, "param"), _cptr(grad, "grad"), _cptr(exp_avg, "exp_avg"),
                                         _cptr(exp_avg_sq, "exp_avg_sq"), param.numel(), lr, beta1, beta2, eps,
                                         weight_decay, grad_scale, int(step), _ptr(lr_dev), _ptr(step_dev),
                                         _stream()), "dstd_adam_step")


_backend = None


def backend():
    """The active backend.  Product code only ever gets the CUDA one; tests may inject the ABI emulation."""
    global _backend
    if _backend is None:
        _backend = CudaBackend()
    return _backend


def _set_backend_for_tests(b):
    global _backend
    prev = _backend
    _backend = b
    return prev
