"""Drop-in module mirrors of the reference model classes, std and fast variants in one place.

Each class keeps the reference's constructor signature, sub-module / parameter names and registration
order (so ``state_dict`` keys, shapes, ordering and RNG consumption at init are identical and reference
checkpoints load with ``strict=True``), but every ``forward`` runs on the sm_100a kernels through
``dstd_gcn_b200.ops``.  The nn.Conv2d / nn.Linear / nn.BatchNorm1d / nn.PReLU members are parameter holders only.

Reference classes mirrored (file:line in /root/reference):
  BatchNorm      model/dstdgcn.py:35-50     model/dstdgcn_fast.py:41-56
  DSTDGC         model/dstdgcn.py:53-94     model/dstdgcn_fast.py:59-155
  DSTDGCB        model/dstdgcn.py:97-163    model/dstdgcn_fast.py:158-275
  ConvTemporalGraphical  :166-188 (legacy, dead in the shipped assembly; kept for API completeness)
  ST_GCNN_layer  model/dstdgcn.py:191-249   model/dstdgcn_fast.py:338-450
  DSTDGCN        model/dstdgcn.py:252-317   model/dstdgcn_fast.py:453-614

Internal activation convention: logical [N,C,T,V] tensors with arbitrary strides.  The fast variant's public
[N,T,V,C] tensors are viewed as logical [N,C,T,V] by a permute (no copy); inside DSTDGCN both variants run
the same channel-major layout and differ only by flags (transposed dynamic adjacency, v*C+c BN order).
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn as nn

from .. import ops
from .layers.graph import Graph
from .layers.time import Time


def conv_init(conv):
    if conv.weight is not None:
        nn.init.kaiming_normal_(conv.weight, mode="fan_out")
    if conv.bias is not None:
        nn.init.constant_(conv.bias, 0)


def bn_init(bn, scale):
    nn.init.constant_(bn.weight, scale)
    nn.init.constant_(bn.bias, 0)


def weights_init(m):
    # same selection rule as the reference (class name contains "Conv"), dstdgcn.py:26-32
    if "Conv" in m.__class__.__name__:
        if hasattr(m, "weight"):
            nn.init.kaiming_normal_(m.weight, mode="fan_out")
        if isinstance(getattr(m, "bias", None), torch.Tensor):
            nn.init.constant_(m.bias, 0)


def _logical(x, fast):
    """public layout -> logical [N,C,T,V] view."""
    return x.permute(0, 3, 1, 2) if fast else x


def _public(x4, fast):
    """logical [N,C,T,V] -> contiguous tensor in the variant's public layout."""
    return (x4.permute(0, 2, 3, 1) if fast else x4).contiguous()


def _w2(w):
    return w if w.dim() == 2 else w.view(w.shape[0], w.shape[1])


class _BatchNormBase(nn.Module):
    _fast = False

    def __init__(self, feature_channels, joint_dim, time_dim):
        super().__init__()
        self.c = feature_channels
        self.v = joint_dim
        self.t = time_dim
        self.bn = nn.BatchNorm1d(feature_channels * joint_dim)

    def forward(self, x):
        x4 = _logical(x, self._fast)
        n, c, t, v = x4.shape
        assert (c, t, v) == (self.c, self.t, self.v)
        out = ops.bn_act(x4, self.bn, vc_order=self._fast)
        return _public(out, self._fast)


class _DSTDGCBase(nn.Module):
    _fast = False

    def __init__(self, in_channels, out_channels, ref_channels, kpt_channels, red_channels=2, mode="spatial"):
        super().__init__()
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.ref_channels = ref_channels
        self.kpt_channels = kpt_channels
        self.red_channels = red_channels
        self.mode = mode
        assert mode in {"spatial", "temporal"}
        if red_channels != 2:
            raise NotImplementedError("the sm_100a kernels implement the reference's red_channels=2")
        self.conv_m1 = nn.Conv2d(in_channels, red_channels, 1)
        self.conv_m2 = nn.Conv2d(in_channels, red_channels, 1)
        self.conv_rm = nn.Conv2d(red_channels * ref_channels, ref_channels, 1)
        self.tanh = nn.Tanh()
        self.conv_f = nn.Linear(in_channels, out_channels) if self._fast else nn.Conv2d(in_channels, out_channels, 1)
        self.init_parameter()

    def init_parameter(self):
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                conv_init(m)

    def branch(self, adj, adj_w=None, adj_r=None):
        """Weight bundle in the layout `ops.gc_unit` expects."""
        return dict(w_m1=self.conv_m1.weight, b_m1=self.conv_m1.bias, w_m2=self.conv_m2.weight,
                    b_m2=self.conv_m2.bias, w_rm=self.conv_rm.weight, b_rm=self.conv_rm.bias,
                    w_f=self.conv_f.weight, b_f=self.conv_f.bias, adj=adj, adj_w=adj_w, adj_r=adj_r)

    def forward(self, x, A=None, alpha_m=1):
        x4 = _logical(x, self._fast)
        k = x4.shape[3] if self.mode == "spatial" else x4.shape[2]
        xu = x4 if self.mode == "spatial" else x4.permute(0, 1, 3, 2)
        if not isinstance(alpha_m, torch.Tensor):
            alpha_m = torch.full((1,), float(alpha_m), dtype=x.dtype, device=x.device)
        adj = A.reshape(k, k).contiguous()
        out = ops.gc_unit(xu, alpha_m.reshape(1), [self.branch(adj)], adj_t=self._fast)
        if self.mode != "spatial":
            out = out.permute(0, 1, 3, 2)
        return _public(out, self._fast)


class _DSTDGCBBase(nn.Module):
    _fast = False
    _gc_cls = _DSTDGCBase
    _bn_cls = _BatchNormBase

    def __init__(self, in_channels, out_channels, time_dim, joint_dim, layout="h36m"):
        super().__init__()
        A_s = Graph(layout).get_all_adjacency()
        A_t = Time(time_dim).get_all_adjacency()
        if not self._fast:
            self.A_s = nn.Parameter(torch.tensor(A_s, dtype=torch.float32), False)
            self.W_s = nn.Parameter(torch.zeros_like(self.A_s))
            # the reference's R_s aliases A_s' storage until the model is moved to the GPU (dstdgcn.py:107-109);
            # this is the post-.to(device) behaviour: an independent copy.
            self.R_s = nn.Parameter(self.A_s.detach().clone())
        else:
            self.A_s = nn.Parameter(torch.tensor(A_s, dtype=torch.float32))
        self.A_t = nn.Parameter(torch.tensor(A_t, dtype=torch.float32), False)
        self.R_t = nn.Parameter(torch.zeros_like(self.A_t))

        self.conv_s = nn.ModuleList()
        self.conv_t = nn.ModuleList()
        if in_channels != out_channels:
            mix = nn.Linear(in_channels, out_channels) if self._fast else nn.Conv2d(in_channels, out_channels, 1)
            self.residual = nn.Sequential(mix, self._bn_cls(out_channels, joint_dim, time_dim))
        else:
            self.residual = lambda x: x
        for _ in range(A_s.shape[0]):
            self.conv_s.append(self._gc_cls(in_channels, out_channels, time_dim, joint_dim, mode="spatial"))
        self.alpha_sm = nn.Parameter(torch.zeros(1))
        self.bn = self._bn_cls(out_channels, joint_dim, time_dim)
        for _ in range(A_t.shape[0]):
            self.conv_t.append(self._gc_cls(out_channels, out_channels, joint_dim, time_dim, mode="temporal"))
        self.alpha_tm = nn.Parameter(torch.zeros(1))
        self.prelu = nn.PReLU()
        self.do = nn.Dropout(0.1)     # never applied, as in the reference (dstdgcn.py:133)

    def init_parameter(self):
        stdt = 1. / math.sqrt(self.R_t.size(1))
        self.R_t.data.uniform_(-stdt, stdt)
        if not self._fast:
            stdt = 1. / math.sqrt(self.R_s.size(1))
            self.R_s.data.uniform_(-stdt, stdt)

    # ---- fused path on logical [N,C,T,V]; returns logical [N,Cout,T,V] held in [N,C,V,T] memory order
    def run(self, x4, skip4=None):
        fast = self._fast
        if isinstance(self.residual, nn.Sequential):
            mix, rbn = self.residual[0], self.residual[1]
            r = ops.bn_act(ops.chmix(x4, _w2(mix.weight), mix.bias), rbn.bn, vc_order=fast)
        else:
            r = x4
        # unbind (backward = one stack) instead of indexing (backward = zeros + copy per branch + a sum)
        a_s = self.A_s.unbind(0)
        if fast:
            brs = [g.branch(a_s[i]) for i, g in enumerate(self.conv_s)]
        else:
            w_s, r_s = self.W_s.unbind(0), self.R_s.unbind(0)
            brs = [g.branch(a_s[i], w_s[i], r_s[i]) for i, g in enumerate(self.conv_s)]
        if ops.FUSE_SKIP_GRAD and ops.FUSE_RES_GRAD and r is x4:
            # chain the consumers of the block input (see ops.FUSE_SKIP_GRAD): the residual reads the alias returned by
            # the spatial unit's node
            same_skip = skip4 is x4
            y, r = ops.gc_unit(x4, self.alpha_sm, brs, adj_t=fast, pass_x=True)
            if same_skip:
                skip4 = r
        else:
            y = ops.gc_unit(x4, self.alpha_sm, brs, adj_t=fast)
        if ops.FUSE_SKIP_GRAD and skip4 is not None and skip4 is r:
            # the block input is both the BN residual and the layer skip: route the skip through the BN node so that
            # the two gradients are summed inside the BN backward kernel
            x2, skip4 = ops.bn_act(y, self.bn.bn, r=r, prelu=self.prelu.weight, vc_order=fast,
                                   out_order=ops.ORDER_V_MAJOR, pass_r=True)
        else:
            x2 = ops.bn_act(y, self.bn.bn, r=r, prelu=self.prelu.weight, vc_order=fast, out_order=ops.ORDER_V_MAJOR)
        a_t, r_t = self.A_t.unbind(0), self.R_t.unbind(0)
        brt = [g.branch(a_t[i], None, r_t[i]) for i, g in enumerate(self.conv_t)]
        skip_u = None if skip4 is None else skip4.permute(0, 1, 3, 2)
        z_u = ops.gc_unit(x2.permute(0, 1, 3, 2), self.alpha_tm, brt, skip_u=skip_u, adj_t=fast)
        return z_u.permute(0, 1, 3, 2)

    def forward(self, x):
        return _public(self.run(_logical(x, self._fast)), self._fast)


class _ConvTemporalGraphicalBase(nn.Module):
    """Legacy STS-GCN style layer (refine=False).  Never built by DSTDGCN; plain torch, not on the hot path."""
    _fast = False

    def __init__(self, time_dim, joints_dim, layout="h36m"):
        super().__init__()
        self.A = nn.Parameter(torch.empty(time_dim, joints_dim, joints_dim))
        stdv = 1. / math.sqrt(self.A.size(1))
        self.A.data.uniform_(-stdv, stdv)
        self.T = nn.Parameter(torch.empty(joints_dim, time_dim, time_dim))
        stdv = 1. / math.sqrt(self.T.size(1))
        self.T.data.uniform_(-stdv, stdv)
        adj = Graph(layout).get_adjacency()[np.newaxis, :]
        self.A_fixed = nn.Parameter(torch.tensor(adj, dtype=torch.float32), requires_grad=False)

    def forward(self, x):
        x = torch.einsum("nctv,vtq->ncqv", (x, self.T))
        x = torch.einsum("nctv,tvw->nctw", (x, self.A + self.A_fixed))
        return x.contiguous()


class _STLayerBase(nn.Module):
    _fast = False
    _blk_cls = _DSTDGCBBase
    _ctg_cls = _ConvTemporalGraphicalBase

    def __init__(self, in_channels, out_channels, kernel_size, stride, time_dim, joints_dim, bias=True, refine=False,
                 residual=True, layout="h36m"):
        super().__init__()
        self.kernel_size = kernel_size
        self.refine = refine
        assert self.kernel_size[0] % 2 == 1
        assert self.kernel_size[1] % 2 == 1
        padding = ((self.kernel_size[0] - 1) // 2, (self.kernel_size[1] - 1) // 2)
        if refine:
            self.stgcn = nn.ModuleList()
            self.stgcn.append(nn.Sequential(self._blk_cls(in_channels, out_channels, time_dim, joints_dim, layout)))
        else:
            self.stgcn = nn.Sequential(
                self._ctg_cls(time_dim, joints_dim, layout),
                nn.Conv2d(in_channels, out_channels, (self.kernel_size[0], self.kernel_size[1]), (stride, stride),
                          padding))
        if not residual:
            self.residual = None
        elif stride != 1 or in_channels != out_channels:
            self.residual = nn.Conv2d(in_channels, out_channels, kernel_size=1, stride=1)
        else:
            self.residual = nn.Identity()
        self.apply(weights_init)

    def run(self, x4):
        """Fused refine=True path on logical [N,C,T,V]: DSTDGCB with the layer skip added in its last kernel."""
        if self.residual is None:
            skip = None
        elif isinstance(self.residual, nn.Identity):
            skip = x4
        else:
            skip = ops.chmix(x4, _w2(self.residual.weight), self.residual.bias)
        y = None
        for i, stb in enumerate(self.stgcn):
            z = stb[0].run(x4, skip if i == 0 else None)
            y = z if y is None else y + z
        return y

    def forward(self, x):
        if self.refine:
            return _public(self.run(_logical(x, self._fast)), self._fast)
        res = self.residual(x) if self.residual is not None else None      # legacy path, plain torch
        x = self.stgcn(x)
        return x + res if res is not None else x


class _DSTDGCNBase(nn.Module):
    _fast = False
    _layer_cls = _STLayerBase
    _bn_cls = _BatchNormBase

    def __init__(self, input_channels, input_time_frame, output_time_frame, st_gcnn_dropout, joints_to_consider,
                 num_feature=64, num_layers=7, layout="h36m"):
        super().__init__()
        self.input_channels = input_channels
        self.input_time_frame = input_time_frame
        self.output_time_frame = output_time_frame
        self.joints_to_consider = joints_to_consider
        self.encoders = nn.ModuleList()
        all_time_frame = input_time_frame + output_time_frame
        self.conv_st_in = self._layer_cls(input_channels, num_feature, [1, 1], 1, all_time_frame, joints_to_consider,
                                          True, True, False, layout)
        self.bn_in = self._bn_cls(num_feature, joints_to_consider, all_time_frame)
        self.do_in = nn.Dropout(st_gcnn_dropout)
        for _ in range(num_layers):
            self.encoders.append(nn.Sequential(
                self._layer_cls(num_feature, num_feature, [1, 1], 1, all_time_frame, joints_to_consider, False, True,
                                True, layout),
                self._bn_cls(num_feature, joints_to_consider, all_time_frame),
                nn.PReLU()))
        self.conv_st_out = self._layer_cls(num_feature, input_channels // 2, [1, 1], 1, all_time_frame,
                                           joints_to_consider, True, True, False, layout)
        self.prelu = nn.PReLU()
        self.dropout_mask = None      # test hook: explicit (already 1/(1-p)-scaled) [N,C,T,V] mask, or a list of masks
        self._mask_calls = 0          # used in turn by consecutive forward calls (the two passes of a training step)

    def _mask(self, n, c, t, v, device):
        if self.dropout_mask is not None:
            if isinstance(self.dropout_mask, (list, tuple)):
                mk = self.dropout_mask[self._mask_calls % len(self.dropout_mask)]
                self._mask_calls += 1
                return mk
            return self.dropout_mask
        if self.training and self.do_in.p > 0:
            # torch's Philox stream draws the mask; applying it is fused into the BN/PReLU kernel
            return self.do_in(torch.ones((n, c, t, v), dtype=torch.float32, device=device))
        return None

    @property
    def coords(self):
        """Coordinates per joint of the input pose x [N, T, V, D]: D = input_channels / 2 (3 for xyz)."""
        return self.input_channels // 2

    def forward(self, x):
        n, t, v, d = x.shape
        assert t == self.input_time_frame + self.output_time_frame
        if self.input_channels != 2 * d:
            # the network reads cat(x, x - x[:, -1:]): 2*D channels (model/dstdgcn.py:298-303)
            raise ValueError(f"input_channels = {self.input_channels} needs x [N, T, V, input_channels / 2]"
                             f"{'' if self.input_channels % 2 else f' = {self.input_channels // 2}'}"
                             f" coordinates per joint; x has {d}")
        if d > ops.MAX_COORDS:
            raise NotImplementedError(f"the head/tail kernels take at most {ops.MAX_COORDS} coordinates per joint "
                                      f"(input_channels <= {2 * ops.MAX_COORDS}); got {d}")
        fast = self._fast
        h = ops.prep(x)
        z = self.conv_st_in.run(h)
        nf = z.shape[1]
        h = ops.bn_act(z, self.bn_in.bn, prelu=self.prelu.weight, mask=self._mask(n, nf, t, v, x.device),
                       vc_order=fast, out_order=ops.ORDER_T_MAJOR)
        for gcn in self.encoders:
            z = gcn[0].run(h)
            h = ops.bn_act(z, gcn[1].bn, prelu=gcn[2].weight, vc_order=fast, out_order=ops.ORDER_T_MAJOR)
        z = self.conv_st_out.run(h)
        return ops.finish(z, x)
