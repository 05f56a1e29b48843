"""User-registered skeletons (``graph.register_layout``) of up to 128 joints, end to end.

CPU: registration and its validation, the adjacency built from a spec, the state_dict of a 38-joint model, ``mirror``
on a registered layout, and the fp64 ABI emulation of BatchNorm at V = 48 against autograd of the oracle.
GPU: every BatchNorm entry point at V = 33 .. 128 against the emulation in fp64, the bulk-copy fast path bit for bit
against the generic kernels, the synchronised phases, whole models against the oracle, Adam steps, the captured step,
and the kernels a pass launches (no silent fall-back to the generic BatchNorm kernels)."""
import numpy as np
import pytest
import torch

from dstd_gcn_b200 import data
from dstd_gcn_b200.model.layers import graph
from oracle import dstd_oracle as orc
from oracle.abi_emul import EmulBackend
from tests.helpers import load_json, max_abs, rel_err

DEV = "cuda"
EM = EmulBackend()


def skeleton_spec(joints):
    """A deterministic tree skeleton: bone (j // 2, j) for every joint j > 0, part pairs (j, j + 2) every third joint,
    mirror pairs (odd, next even) joints."""
    bones = [(j // 2, j) for j in range(1, joints)]
    parts = [(j, j + 2) for j in range(0, joints - 2, 3)]
    right = list(range(1, joints - 1, 2))
    return dict(joints=joints, bones=bones, parts=parts, mirror=(right, [k + 1 for k in right]))


def layout(joints, mirror=True):
    """Name of a registered synthetic skeleton of `joints` joints (registered on first use)."""
    name = f"test_skel{joints}" + ("" if mirror else "_nomirror")
    if name not in graph._EDGES:
        sp = skeleton_spec(joints)
        graph.register_layout(name, sp["joints"], sp["bones"], sp["parts"], sp["mirror"] if mirror else None)
    return name


# ====================================================================================================== CPU
def test_register_and_use_by_name():
    name = layout(38)
    g = graph.Graph(name)
    assert g.num_joint == 38 and g.layout == name
    assert g.bone_pair == [list(e) for e in skeleton_spec(38)["bones"]]
    with pytest.raises(NotImplementedError):
        graph.Graph("no_such_layout")


@pytest.mark.parametrize("kw,match", [
    (dict(joints=0), "joints"),
    (dict(joints=129), "joints"),
    (dict(joints=3.0), "int"),
    (dict(bones=[(2, 1)]), "0 <= i < j"),
    (dict(bones=[(1, 1)]), "self loop"),
    (dict(bones=[(0, 5)]), "0 <= i < j"),
    (dict(bones=[(-1, 2)]), "0 <= i < j"),
    (dict(bones=[(0, 1), (0, 1)]), "duplicate"),
    (dict(parts=[(0, 2), (0, 2)]), "duplicate"),
    (dict(parts=[(0, 1, 2)]), "pair"),
    (dict(mirror=([1, 2], [3])), "right has"),
    (dict(mirror=([1, 2], [2, 3])), "disjoint"),
    (dict(mirror=([1, 1], [2, 3])), "disjoint"),
    (dict(mirror=([1], [2], [3])), "pair"),
    (dict(mirror=([-1], [2])), "negative"),
])
def test_register_validation(kw, match):
    args = dict(name="test_invalid", joints=5, bones=[(0, 1), (1, 2)], parts=[(0, 3)], mirror=None)
    args.update(kw)
    with pytest.raises((ValueError, TypeError), match=match):
        graph.register_layout(**args)
    assert "test_invalid" not in graph._EDGES


def test_register_refuses_existing_names():
    for name in ("h36m", "cmu", "3dpw", layout(33)):
        with pytest.raises(ValueError, match="already registered"):
            graph.register_layout(name, 5, [(0, 1)], [])
    with pytest.raises(ValueError, match="name"):
        graph.register_layout("", 5, [(0, 1)], [])


def test_adjacency_from_spec():
    for v in (1, 33, 55, 128):
        sp = skeleton_spec(v)
        a = graph.Graph(layout(v)).get_all_adjacency()
        assert a.shape == (2, v, v) and a.dtype == np.float64
        conn, part = a
        assert np.array_equal(conn, conn.T) and np.array_equal(part, part.T)
        assert np.array_equal(np.diag(conn), np.ones(v)) and np.array_equal(np.diag(part), np.zeros(v))
        ref_c, ref_p = np.eye(v), np.zeros((v, v))
        for i, j in sp["bones"]:
            ref_c[i, j] = ref_c[j, i] = 1
        for i, j in sp["parts"]:
            ref_p[i, j] = ref_p[j, i] = 1
        assert np.array_equal(conn, ref_c) and np.array_equal(part, ref_p)


@pytest.mark.parametrize("variant,golden,v0", [("std", "std_cmu", 25), ("fast", "fast_h36m", 22)])
def test_state_dict_of_38_joint_model(variant, golden, v0):
    """The keys of the reference's model (25-joint CMU for std, 22-joint H3.6M for fast), with every joint-sized
    dimension at 38: A_s [2,V,V], the temporal conv_rm [V, 2V], BatchNorm over C*V channels."""
    from dstd_gcn_b200.model import dstdgcn, dstdgcn_fast
    mod = dstdgcn if variant == "std" else dstdgcn_fast
    spec = load_json("state_keys.json")[golden]
    assert spec["args"][4] == v0 and spec["args"][5] == 64
    m = mod.DSTDGCN(6, 10, 25, 0.1, 38, 64, 5, layout(38))
    sd = m.state_dict()
    scale = {v0: 38, 2 * v0: 76, 64 * v0: 64 * 38, 3 * v0: 3 * 38}
    assert list(sd) == [k for k, *_ in spec["keys"]]
    for k, shape, *_ in spec["keys"]:
        assert list(sd[k].shape) == [scale.get(d, d) for d in shape], k
    assert torch.equal(sd["encoders.0.0.stgcn.0.0.A_s"],
                       torch.from_numpy(graph.Graph(layout(38)).get_all_adjacency()).float())


def test_mirror_on_registered_layout():
    sp = skeleton_spec(38)
    g = torch.Generator().manual_seed(4)
    x = torch.randn(3, 7, 38 * 3, generator=g)
    got = data.mirror(x, layout(38))
    a = x.numpy().reshape(3, 7, 38, 3)
    ref = a.copy()
    right, left = sp["mirror"]
    ref[:, :, right] = a[:, :, left]
    ref[:, :, left] = a[:, :, right]
    ref[..., 0] *= -1
    assert np.array_equal(got.numpy(), ref.reshape(3, 7, 38 * 3))
    with pytest.raises(ValueError, match="without mirror lists"):
        data.mirror(x, layout(38, mirror=False))
    (b,) = list(data.DevicePrefetcher([x], 3, 4, device="cpu", mirror_layout=layout(38)))
    assert torch.equal(b[3], torch.cat((x, got)))         # the mirrored copy is appended to the batch


@pytest.mark.parametrize("vc,use_r,use_prelu,use_mask,training",
                         [(False, True, True, False, True), (True, False, False, True, True),
                          (False, True, True, True, False)], ids=["res_prelu", "vc_mask", "eval"])
def test_emulated_bn_at_48_joints_vs_oracle_autograd(vc, use_r, use_prelu, use_mask, training):
    """The fp64 ABI emulation (the GPU tests' yardstick) at V = 48 against torch autograd through the oracle's
    BatchNorm + residual + PReLU + mask."""
    n, c, t, v = 3, 4, 6, 48
    g = torch.Generator().manual_seed(48)
    y = torch.randn(n, c, t, v, generator=g, dtype=torch.float64) * 2 + 3
    r = torch.randn(n, c, t, v, generator=g, dtype=torch.float64) if use_r else None
    gamma = torch.randn(c * v, generator=g, dtype=torch.float64) * 0.5 + 1
    beta = torch.randn(c * v, generator=g, dtype=torch.float64) * 0.5
    rm = torch.randn(c * v, generator=g, dtype=torch.float64) * 0.5
    rv = torch.rand(c * v, generator=g, dtype=torch.float64) + 0.5
    prelu = torch.tensor([0.25], dtype=torch.float64) if use_prelu else None
    mask = (torch.rand(n, c, t, v, generator=g) > 0.1).double() / 0.9 if use_mask else None
    gout = torch.randn(n, c, t, v, generator=g, dtype=torch.float64)
    out_e, mean_e, istd_e = EM.bn_act_forward(y, r, gamma, beta, rm.clone(), rv.clone(), None, prelu, mask, vc,
                                              training, 1e-5, 0.1)
    gy_e, gr_e, gg_e, gb_e, gp_e = EM.bn_act_backward(y, r, gout, gamma, beta, prelu, mask, mean_e, istd_e, vc,
                                                      training, True)

    # the oracle's BatchNorm: [N,C,T,V] with channel c*V+v, or (fast) [N,T,V,C] with channel v*C+c = the vc order
    yl = y.clone().requires_grad_(True)
    rl = r.clone().requires_grad_(True) if use_r else None
    p = {"bn.weight": gamma.clone().requires_grad_(True), "bn.bias": beta.clone().requires_grad_(True),
         "bn.running_mean": rm.clone(), "bn.running_var": rv.clone()}
    al = prelu.clone().requires_grad_(True) if use_prelu else None
    h = orc.batchnorm(yl.permute(0, 2, 3, 1) if vc else yl, p, "", training, fast=vc)
    h = h.permute(0, 3, 1, 2) if vc else h
    if use_r:
        h = h + rl
    if use_prelu:
        h = orc.prelu(h, al)
    if use_mask:
        h = h * mask
    h.backward(gout)
    assert max_abs(out_e, h) < 1e-12
    assert max_abs(gy_e, yl.grad) < 1e-10
    assert max_abs(gg_e, p["bn.weight"].grad) < 1e-10 and max_abs(gb_e, p["bn.bias"].grad) < 1e-10
    if use_r:
        assert max_abs(gr_e, rl.grad) < 1e-12
    if use_prelu:
        assert abs(float(gp_e) - float(al.grad)) < 1e-10 * max(1.0, abs(float(al.grad)))


# ====================================================================================================== GPU
def _be():
    from dstd_gcn_b200 import _lib
    b = _lib.backend()
    assert b.name == "cuda"
    return b


def _ordered(g, n, c, t, v, order):
    if order == "t":
        return torch.randn((n, c, t, v), generator=g, dtype=torch.float64)
    return torch.randn((n, c, v, t), generator=g, dtype=torch.float64).permute(0, 1, 3, 2)


def _to_dev(t):
    if t is None:
        return None
    out = torch.empty_strided(t.shape, t.stride(), dtype=torch.float32, device=DEV)
    out.copy_(t.float())
    return out


# n, c, t, v, y_order, r_order, out_order, vc, prelu, mask, training   (fast = the fast path takes the shape)
BN_CASES = [
    (4, 8, 35, 33, "t", "t", 2, False, True, False, True),      # odd T*V, 4-channel slab of 4620: generic
    (4, 8, 35, 38, "v", None, 1, False, True, True, True),      # input BN with dropout mask: generic
    (3, 8, 35, 38, "t", "t", 2, True, True, False, True),       # vc order, block BN: fast (2-channel slab)
    (40, 16, 35, 38, "v", None, 1, False, True, False, True),   # more samples than splits
    (3, 8, 35, 55, "v", "v", 0, False, True, False, False),     # eval
    (5, 4, 35, 64, "t", "t", 2, False, True, False, True),      # fast, 1-channel slab
    (3, 4, 35, 64, "t", None, 0, True, False, False, False),    # eval, plain BatchNorm, vc order
    (4, 4, 35, 128, "t", "t", 2, False, True, False, True),     # fast BIG: 4480 positions
    (3, 4, 32, 128, "v", None, 1, False, True, True, True),     # mask at V = 128: generic, T*V = 4096
    (3, 4, 32, 128, "t", "t", 2, True, True, False, False),     # eval, vc order
    (2, 3, 2, 100, "t", "t", 2, False, True, False, True),      # tiny T: fewer positions per plane than joints
]


@pytest.mark.gpu
@pytest.mark.parametrize("fast", ["1", "0"])
@pytest.mark.parametrize("case", BN_CASES, ids=[str(i) for i in range(len(BN_CASES))])
def test_bn_act_abi_wide(case, fast, monkeypatch):
    n, c, t, v, yo, ro, out_order, vc, use_prelu, use_mask, training = case
    if fast == "0" and t * v > 4096:
        pytest.skip("the generic kernels run up to 4096 positions")
    monkeypatch.setenv("DSTD_BN_FAST", fast)
    from dstd_gcn_b200.ops import _out_like
    g = torch.Generator().manual_seed(n * 13 + c + v)
    be = _be()
    y = _ordered(g, n, c, t, v, yo) * 2.0 + 3.0
    r = _ordered(g, n, c, t, v, ro) if ro else None
    gamma, beta = torch.randn(c * v, generator=g, dtype=torch.float64) * 0.5 + 1.0, \
        torch.randn(c * v, generator=g, dtype=torch.float64) * 0.5
    rm, rv = torch.randn(c * v, generator=g, dtype=torch.float64) * 0.5, \
        torch.rand(c * v, generator=g, dtype=torch.float64) + 0.5
    nbt = torch.tensor(3, dtype=torch.int64)
    prelu = torch.tensor([0.25], dtype=torch.float64) if use_prelu else None
    mask = ((torch.rand((n, c, t, v), generator=g) > 0.1).double() / 0.9) if use_mask else None
    ol = _out_like(y, out_order)
    rm_r, rv_r, nbt_r = rm.clone(), rv.clone(), nbt.clone()
    out_r, mean_r, istd_r = EM.bn_act_forward(y, r, gamma, beta, rm_r, rv_r, nbt_r, prelu, mask, vc, training, 1e-5,
                                              0.1, ol if out_order else None)
    yd, rd = _to_dev(y), _to_dev(r)
    gd, bd, rmd, rvd, nbd = _to_dev(gamma), _to_dev(beta), _to_dev(rm), _to_dev(rv), nbt.to(DEV)
    pd_, md = _to_dev(prelu), _to_dev(mask)
    old = _out_like(yd, out_order)
    out, mean, istd = be.bn_act_forward(yd, rd, gd, bd, rmd, rvd, nbd if training else None, pd_, md, vc, training,
                                        1e-5, 0.1, old if out_order else None)
    torch.cuda.synchronize()
    assert be.lib.dstd_device_error(0) == 0
    assert out.stride() == out_r.stride()
    assert max_abs(out, out_r) < 2e-5 * max(1.0, float(out_r.abs().max()))
    assert max_abs(mean, mean_r) < 1e-5 and rel_err(istd, istd_r) < 1e-5
    if training:
        assert max_abs(rmd, rm_r) < 1e-5 and max_abs(rvd, rv_r) < 1e-5 and int(nbd) == int(nbt_r)
    gout = torch.empty_strided(out_r.shape, out_r.stride(), dtype=torch.float64)
    gout.copy_(torch.randn(tuple(out_r.shape), generator=g, dtype=torch.float64))
    res_r = EM.bn_act_backward(y, r, gout, gamma, beta, prelu, mask, mean_r, istd_r, vc, training, True)
    res = be.bn_act_backward(yd, rd, _to_dev(gout), gd, bd, pd_, md, mean, istd, vc, training, True)
    torch.cuda.synchronize()
    for nm, a, b in zip(("gy", "gr", "ggamma", "gbeta", "gprelu"), res, res_r):
        if b is None:
            assert a is None, nm
            continue
        assert a.shape == b.shape, nm
        assert max_abs(a, b) < 1e-4 * max(1.0, float(b.abs().max())), nm
    if r is not None:
        gadd = torch.empty_strided(out_r.shape, out_r.stride(), dtype=torch.float64)
        gadd.copy_(torch.randn(tuple(out_r.shape), generator=g, dtype=torch.float64))
        res2 = be.bn_act_backward(yd, rd, _to_dev(gout), gd, bd, pd_, md, mean, istd, vc, training, True, _to_dev(gadd))
        torch.cuda.synchronize()
        assert max_abs(res2[1], res_r[1] + gadd) < 1e-4 * max(1.0, float(res_r[1].abs().max()))
        assert res2[1].stride() == res[1].stride()
        assert torch.equal(res2[0], res[0]) and torch.equal(res2[2], res[2]) and torch.equal(res2[3], res[3])


@pytest.mark.gpu
def test_bn_limits_name_the_generic_position_limit():
    """T*V above 4096 runs only where the fast path takes every pass: not with a dropout mask, not with
    DSTD_BN_FAST=0, never for V <= 32.  V above 128 is refused."""
    be = _be()
    g = torch.Generator().manual_seed(1)

    def fwd(c, t, v, mask=False):
        y = _to_dev(_ordered(g, 2, c, t, v, "t"))
        ones, zeros = torch.ones(c * v, device=DEV), torch.zeros(c * v, device=DEV)
        mk = torch.ones(2, c, t, v, device=DEV) if mask else None
        return be.bn_act_forward(y, None, ones, zeros, None, None, None, None, mk, False, True, 1e-5, 0.1)

    fwd(4, 35, 128)
    with pytest.raises(RuntimeError, match="4096 positions"):
        fwd(4, 35, 128, mask=True)
    with pytest.raises(RuntimeError, match="4096 positions"):
        fwd(4, 140, 32)
    with pytest.raises(RuntimeError, match="max 128"):
        fwd(4, 4, 129)


# n, c, t, v, y_order, r_order, out_order, prelu, training
BN_FAST_CASES = [
    (37, 8, 35, 38, "t", "t", 2, True, True),     # 1330 floats: two channels per slab, ragged splits
    (9, 8, 35, 38, "v", None, 1, True, True),     # layer BN
    (5, 8, 35, 64, "t", "t", 2, True, True),      # 2240: one channel per slab
    (5, 8, 35, 64, "v", None, 1, True, False),    # eval
    (5, 4, 35, 128, "t", "t", 2, True, True),     # 4480: BIG
    (3, 4, 35, 128, "v", None, 1, True, True),
    (3, 8, 35, 55, "t", "t", 2, True, True),      # odd plane, 4-channel slab of 7700 > 4096: generic on both sides
    (4, 8, 36, 33, "t", None, 0, False, True),    # 1188: one channel, no PReLU
    (4, 6, 10, 45, "t", "t", 2, True, True),      # 450: two channels
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", BN_FAST_CASES, ids=[str(i) for i in range(len(BN_FAST_CASES))])
def test_bn_fast_path_equals_generic_wide(case, monkeypatch):
    """The wide bulk-copy kernels against the wide generic ones: same arithmetic and summation order, so everything
    but the PReLU-slope gradient is bit-identical; a repeated call gives the same bits.  At T*V > 4096 only the fast
    path runs, and is compared with the fp64 emulation instead."""
    n, c, t, v, yo, ro, out_order, use_prelu, training = case
    g = torch.Generator().manual_seed(n * 7 + c + v)
    be = _be()
    from dstd_gcn_b200.ops import _out_like
    y = _to_dev(_ordered(g, n, c, t, v, yo) * 2.0 + 3.0)
    r = _to_dev(_ordered(g, n, c, t, v, ro)) if ro else None
    gamma, beta = _to_dev(torch.randn(c * v, generator=g, dtype=torch.float64) * 0.5 + 1.0), \
        _to_dev(torch.randn(c * v, generator=g, dtype=torch.float64) * 0.5)
    prelu = _to_dev(torch.tensor([0.25], dtype=torch.float64)) if use_prelu else None
    ol = _out_like(y, out_order)
    res = {}
    flags = ("1", "1again") if t * v > 4096 else ("0", "1", "1again")
    for flag in flags:
        monkeypatch.setenv("DSTD_BN_FAST", flag[0])
        rm, rv = torch.zeros(c * v, device=DEV), torch.ones(c * v, device=DEV)
        nbt = torch.zeros((), dtype=torch.int64, device=DEV)
        out, mean, istd = be.bn_act_forward(y, r, gamma, beta, rm, rv, nbt if training else None, prelu, None, False,
                                            training, 1e-5, 0.1, ol if out_order else None)
        gout = torch.empty_like(out)
        gout.copy_(_to_dev(torch.randn(tuple(out.shape), generator=torch.Generator().manual_seed(5),
                                       dtype=torch.float64)))
        bw = be.bn_act_backward(y, r, gout, gamma, beta, prelu, None, mean, istd, False, training, r is not None)
        bw2 = None
        if r is not None:
            gadd = torch.empty_like(out)
            gadd.copy_(_to_dev(torch.randn(tuple(out.shape), generator=torch.Generator().manual_seed(6),
                                           dtype=torch.float64)))
            bw2 = be.bn_act_backward(y, r, gout, gamma, beta, prelu, None, mean, istd, False, training, True, gadd)
        torch.cuda.synchronize()
        assert be.lib.dstd_device_error(0) == 0
        res[flag] = (out, mean, istd, rm, rv, bw, bw2)
    pairs = [("1", "1again")] + ([("0", "1")] if "0" in res else [])
    for fa, fb in pairs:
        a, b = res[fa], res[fb]
        for i in range(5):
            assert torch.equal(a[i], b[i]), (fa, fb, i)
        for bwa, bwb in ((a[5], b[5]), (a[6], b[6])):
            if bwa is None:
                continue
            for nm, ta, tb in zip(("gy", "gr", "ggamma", "gbeta"), bwa, bwb):
                if ta is None:
                    assert tb is None
                    continue
                assert ta.stride() == tb.stride() and torch.equal(ta, tb), (fa, fb, nm)
            if bwa[4] is not None:
                exact = fa == "1" and fb == "1again"
                assert (torch.equal(bwa[4], bwb[4]) if exact
                        else max_abs(bwa[4], bwb[4]) <= 1e-5 * max(1.0, float(bwa[4].abs().max())))
    if "0" not in res:       # the fast path alone: against the fp64 emulation
        out, mean, istd = res["1"][:3]
        y64 = y.double().cpu()
        out_r, mean_r, istd_r = EM.bn_act_forward(y64, r.double().cpu() if r is not None else None, gamma.double().cpu(),
                                                  beta.double().cpu(), None, None, None,
                                                  prelu.double().cpu() if prelu is not None else None, None, False,
                                                  True, 1e-5, 0.1)
        assert max_abs(out, out_r) < 2e-5 * max(1.0, float(out_r.abs().max()))
        assert max_abs(mean, mean_r) < 1e-5 and rel_err(istd, istd_r) < 1e-5


SYNC_CASES = {
    # name: (shard sizes, c, t, v, y_order, r_order, vc_order, prelu, mask)
    "v38_block": ([2, 3], 8, 35, 38, "t", "t", False, True, False),
    "v38_mask": ([2, 2], 8, 35, 38, "v", None, False, True, True),
    "v55_block": ([1, 3], 4, 35, 55, "t", "t", False, True, False),
    "v55_vc": ([2, 1], 4, 35, 55, "t", None, True, False, False),
    "v38_unequal": ([1, 6, 2], 8, 35, 38, "t", "t", False, True, False),
}


@pytest.mark.gpu
@pytest.mark.parametrize("fast", ["1", "0"])
@pytest.mark.parametrize("name", list(SYNC_CASES))
def test_sync_phases_wide_equal_plain_call(name, fast, monkeypatch):
    """The synchronised-BN phases on shards against one plain call on the concatenated batch (single GPU)."""
    from tests.test_sync_bn import _sync_bn_vs_plain
    monkeypatch.setenv("DSTD_BN_FAST", fast)
    shards, c, t, v, yo, ro, vc, use_prelu, use_mask = SYNC_CASES[name]
    be = _be()
    plain, sync = _sync_bn_vs_plain(be, shards, c, t, v, yo, ro, vc, use_prelu, use_mask, DEV, torch.float32,
                                    sum(shards) * 31 + c + v, check_twice=True)
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


@pytest.mark.gpu
@pytest.mark.parametrize("variant,v,c,layers,n,seed", [("std", 33, 64, 5, 4, 1234), ("fast", 33, 64, 5, 4, 99),
                                                       ("std", 38, 64, 5, 4, 1234), ("fast", 38, 64, 5, 4, 99),
                                                       ("std", 55, 32, 3, 2, 1234), ("fast", 55, 32, 3, 2, 7)])
def test_model_vs_oracle_wide(variant, v, c, layers, n, seed):
    """Whole models on registered skeletons against the fp64 oracle, with the gates of the full-size check in
    test_gpu_parity.py: the fp32 oracle (the reference's own arithmetic) is the yardstick.  V = 33 and 38 run the fused
    unit kernels, V = 55 the shape-generic ones (smaller C, L and batch).

    The gates compare one rounding realisation with another, so an input at which a pre-activation sits on a PReLU or
    ReLU-like kink within rounding distance makes either side jump by 1e-3 .. 1e-2 in dx.  Such inputs occur for any
    fp32 implementation: at the fast variant's seed 1234, torch's fp32 oracle itself jumps at V = 31 and 48 with one
    ulp of input perturbation, and this library at V = 40 and 55, while every neighbouring joint count stays at the
    fp32 level (1e-5 at C = 32, L = 3).  The inputs used here are not at such a point for either side."""
    fast = variant == "fast"
    tin, tout = 10, 25
    torch.manual_seed(777)
    m = _perturbed(_mod(variant).DSTDGCN(6, tin, tout, 0.0, v, c, layers, layout(v)))
    x = torch.randn(n, tin + tout, v, 3, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)

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
        d = p.grad.double().cpu() - g64[k]
        num += float((d * d).sum())
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


def _batches(n, v, steps, seed):
    import bench
    return [bench.synthetic_batch(n, 35, v, 10, seed=seed + s) for s in range(steps)]


@pytest.mark.gpu
def test_train_steps_38_joints_vs_oracle():
    """Three Adam steps of DSTDGCN(6, 10, 25, 0.1, 38, 64, 5, <38-joint layout>) through TrainStep (inverse pass, with
    the same dropout masks as the oracle) against the fp64 oracle's trajectory, gated like the full-size dropout test."""
    from dstd_gcn_b200.engine import TrainStep
    n, v, c, drop, steps = 32, 38, 64, 0.1, 3
    torch.manual_seed(777)
    m = _perturbed(_mod("std").DSTDGCN(6, 10, 25, drop, v, c, 5, layout(v)))
    g = torch.Generator().manual_seed(99)
    masks = [[(torch.rand(n, c, 35, v, generator=g) >= drop).float() / (1.0 - drop) for _ in range(2)]
             for _ in range(steps)]
    batches = _batches(n, v, steps, 500)

    def oracle_trajectory(dtype):
        p = orc.state_from_module(m, dtype)
        opt = torch.optim.Adam([x for x in p.values() if x.requires_grad], lr=3e-3)
        out = []
        for s in range(steps):
            a, b, tg = (x.to(dtype) for x in batches[s])
            loss = orc.train_loss(p, a, b, tg, dropout_masks=tuple(mk.to(dtype) for mk in masks[s]))
            opt.zero_grad()
            loss.backward()
            opt.step()
            out.append(float(loss.detach()))
        return out

    ref, ref32 = oracle_trajectory(torch.float64), oracle_trajectory(torch.float32)
    md = m.to(DEV).train()
    step = TrainStep(md, lr=3e-3, inverse=True)
    got = []
    for s in range(steps):
        md.dropout_mask = [mk.to(DEV) for mk in masks[s]]
        md._mask_calls = 0
        got.append(float(step(*(x.to(DEV) for x in batches[s]))))
    ref_t, got_t, r32_t = (torch.tensor(x, dtype=torch.float64) for x in (ref, got, ref32))
    dev, dev32 = (got_t - ref_t).abs() / ref_t.abs(), (r32_t - ref_t).abs() / ref_t.abs()
    assert float(dev[0]) < 1e-4, (got, ref)
    assert bool((dev <= torch.clamp(4 * dev32, min=1e-3)).all()), (got, ref, ref32)


@pytest.mark.gpu
def test_captured_step_equals_eager_38_joints():
    """TrainStep.capture() on a 38-joint model: the replayed graph gives the eager trajectory."""
    from dstd_gcn_b200.engine import TrainStep
    v = 38
    batches = [tuple(x.to(DEV) for x in b) for b in _batches(16, v, 3, 40)]

    def fresh():
        torch.manual_seed(5)
        m = _perturbed(_mod("std").DSTDGCN(6, 10, 25, 0.0, v, 16, 2, layout(v))).to(DEV).train()
        return m, TrainStep(m, lr=3e-3, inverse=True)

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


def _bn_kernels(v, lay):
    """BatchNorm kernels launched by one training forward + backward of the bench-shaped model (C=64, L=5, dropout
    0.1), names cut at '<' and without 'dstd::'."""
    from torch.profiler import ProfilerActivity, profile
    torch.manual_seed(3)
    m = _perturbed(_mod("std").DSTDGCN(6, 10, 25, 0.1, v, 64, 5, lay)).to(DEV).train()
    x = torch.randn(8, 35, v, 3, device=DEV)
    m(x).pow(2).mean().backward()                   # warm-up
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        m(x).pow(2).mean().backward()
        torch.cuda.synchronize()
    evs = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "dstd::bn" in e.name),
                 key=lambda e: e.time_range.start)
    return [e.name.removeprefix("void ").removeprefix("dstd::").split("(")[0].split("<")[0] for e in evs]


@pytest.mark.gpu
@pytest.mark.parametrize("v,v_ref", [(38, 22), (64, 24)])
def test_wide_passes_run_the_fast_bn_kernels(v, v_ref):
    """At V = 38 and 64 every BatchNorm the fast-path rules admit runs the bulk-copy `bnf_*_wide` kernels: the launch
    list is that of a <= 32-joint model whose planes take the same slab rule (V = 22: two channels per slab, as at 38;
    V = 24: one channel, as at 64), with the wide twins.  Only the input BN, which carries the dropout mask, and BNs
    whose channel count the slab does not divide run the generic kernels, at both sizes."""
    ref = _bn_kernels(v_ref, "h36m" if v_ref == 22 else layout(v_ref))
    got = _bn_kernels(v, layout(v))
    assert got == [k.replace("_kernel", "_wide_kernel") if k.startswith(("bnf_", "bn_apply", "bn_bwd_apply"))
                   else k for k in ref]
    applies = [k for k in got if k.startswith(("bnf_apply", "bn_apply"))]
    assert applies.count("bnf_apply_wide_kernel") >= 12 and "bn_apply_wide_kernel" in applies, applies
