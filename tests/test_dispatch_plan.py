"""Kernel-path and workspace decisions of the DSTD-GC entry points.

Without a GPU: whether a call keeps ``xa``, and the workspace sizes of every entry point, for the unit shapes of the
parity tests and a (P, K) sweep across the 40-wide specialised tiles, under the default switches and each documented
switch setting (set in-process: the library reads them per call).  The sizes and the xa decision do not depend on the
switches, so a caller that sized its buffers before flipping one still hands over enough workspace.

On the GPU: the kernels one forward + backward launches, per shape and switch setting; and the BatchNorm kernels
(with template arguments, grid, block and dynamic shared memory) of the BN parity cases, with the fast path on and off.

TABLE and KERNELS hold what the library did before these decisions were moved into one plan (api.cu gc_plan), and
BN_LAUNCHES what it did before the BatchNorm dispatch macros became templates (bn_act.cu with_u / with_nj / with_bnf);
a change to any of them is a change of what the library computes, allocates or launches."""
import pytest
import torch

import __graft_entry__ as entry
from dstd_gcn_b200 import _lib
from tests import test_gpu_parity as gp
from tests.test_gpu_parity import GC_CASES, STRESS_CASES

SETTINGS = {
    "default": {},
    "unit_tc": {"DSTD_UNIT_TC": "1"},
    "bf16": {"DSTD_PRECISION": "bf16"},
    "disable_tc": {"DSTD_DISABLE_TC": "1"},
    "bgemm_cuda_core": {"DSTD_BGEMM_TC": "0"},
}

_PK = (1, 22, 39, 40, 41, 48, 64, 125, 128)
SHAPES = list(dict.fromkeys([c[:6] for c in GC_CASES + STRESS_CASES] + [(4, 64, 64, p, k, 2) for p in _PK for k in _PK]))

TABLE = {
    # (n, cin, cout, p, k, nb): (needs_xa, gc_fwd_ws, gc_bwd_ws, chmix_bwd_ws, bn_act_ws)
    (3, 6, 16, 35, 22, 2): (0, 60672, 941056, 2560, 8960),
    (2, 16, 16, 22, 35, 1): (0, 34816, 691456, 4608, 9472),
    (2, 64, 64, 35, 22, 2): (0, 207872, 11037184, 66816, 23296),
    (2, 64, 64, 22, 35, 1): (0, 104448, 5538304, 66816, 36608),
    (2, 16, 3, 40, 23, 2): (0, 65536, 797440, 1280, 1792),
    (2, 3, 3, 25, 35, 1): (0, 30208, 355840, 512, 2304),
    (2, 8, 8, 12, 22, 2): (0, 62720, 435712, 1024, 3328),
    (1, 5, 7, 3, 4, 1): (0, 30208, 108288, 512, 768),
    (5, 64, 64, 40, 23, 2): (0, 207872, 11813632, 150016, 60416),
    (1, 6, 24, 125, 22, 2): (1, 64000, 2751232, 4352, 4864),
    (2, 24, 24, 22, 125, 1): (1, 33792, 26391808, 26880, 48640),
    (1, 72, 80, 125, 22, 2): (1, 152064, 18717696, 140544, 14848),
    (1, 16, 3, 22, 125, 1): (1, 29696, 12836096, 1536, 3584),
    (2, 130, 136, 35, 22, 2): (1, 815360, 46557952, 285440, 49408),
    (1, 256, 256, 125, 22, 2): (1, 2029312, 170805504, 1579264, 46336),
    (1, 256, 256, 22, 125, 1): (1, 1028864, 96957952, 1579264, 257280),
    (4, 64, 64, 1, 1, 2): (0, 207872, 10669824, 16896, 3328),
    (4, 64, 64, 1, 22, 2): (0, 207872, 10703104, 16896, 46336),
    (4, 64, 64, 1, 39, 2): (0, 207872, 10771968, 16896, 81152),
    (4, 64, 64, 1, 40, 2): (0, 207872, 10776576, 16896, 83200),
    (4, 64, 64, 1, 41, 2): (1, 124672, 11638784, 16896, 85248),
    (4, 64, 64, 1, 48, 2): (1, 124672, 12727808, 16896, 99584),
    (4, 64, 64, 1, 64, 2): (1, 124672, 15303680, 16896, 132352),
    (4, 64, 64, 1, 125, 2): (1, 124672, 74994688, 16896, 257280),
    (4, 64, 64, 1, 128, 2): (1, 124672, 79682560, 16896, 263424),
    (4, 64, 64, 22, 1, 2): (0, 207872, 10704384, 16896, 3328),
    (4, 64, 64, 22, 22, 2): (0, 207872, 11118848, 66816, 46336),
    (4, 64, 64, 22, 39, 2): (0, 207872, 11930112, 116736, 81152),
    (4, 64, 64, 22, 40, 2): (0, 207872, 11990784, 116736, 83200),
    (4, 64, 64, 22, 41, 2): (1, 124672, 16115456, 133376, 85248),
    (4, 64, 64, 22, 48, 2): (1, 124672, 19074304, 150016, 99584),
    (4, 64, 64, 22, 64, 2): (1, 124672, 25119744, 183296, 132352),
    (4, 64, 64, 22, 125, 2): (1, 124672, 116937216, 366336, 257280),
    (4, 64, 64, 22, 128, 2): (1, 124672, 123389440, 366336, 263424),
    (4, 64, 64, 39, 1, 2): (0, 207872, 10774272, 16896, 3328),
    (4, 64, 64, 39, 22, 2): (0, 207872, 11497216, 116736, 46336),
    (4, 64, 64, 39, 39, 2): (0, 207872, 12909568, 199936, 81152),
    (4, 64, 64, 39, 40, 2): (0, 207872, 13015296, 216576, 83200),
    (4, 64, 64, 39, 41, 2): (1, 124672, 20296704, 216576, 85248),
    (4, 64, 64, 39, 48, 2): (1, 124672, 25188352, 249856, 99584),
    (4, 64, 64, 39, 64, 2): (1, 124672, 34419200, 333056, 132352),
    (4, 64, 64, 39, 125, 2): (1, 124672, 156059136, 649216, 257280),
    (4, 64, 64, 39, 128, 2): (1, 124672, 164063232, 649216, 263424),
    (4, 64, 64, 40, 1, 2): (0, 207872, 10779136, 16896, 3328),
    (4, 64, 64, 40, 22, 2): (0, 207872, 11520256, 116736, 46336),
    (4, 64, 64, 40, 39, 2): (0, 207872, 12967936, 216576, 81152),
    (4, 64, 64, 40, 40, 2): (0, 207872, 13076480, 216576, 83200),
    (4, 64, 64, 40, 41, 2): (1, 124672, 20548608, 216576, 85248),
    (4, 64, 64, 40, 48, 2): (1, 124672, 25563904, 249856, 99584),
    (4, 64, 64, 40, 64, 2): (1, 124672, 34985472, 333056, 132352),
    (4, 64, 64, 40, 125, 2): (1, 124672, 158503936, 665856, 257280),
    (4, 64, 64, 40, 128, 2): (1, 124672, 166603264, 665856, 263424),
    (4, 64, 64, 41, 1, 2): (1, 207872, 10906624, 16896, 3328),
    (4, 64, 64, 41, 22, 2): (1, 207872, 14472704, 133376, 46336),
    (4, 64, 64, 41, 39, 2): (1, 207872, 20007168, 216576, 81152),
    (4, 64, 64, 41, 40, 2): (1, 207872, 20532992, 216576, 83200),
    (4, 64, 64, 41, 41, 2): (1, 124672, 20836864, 233216, 85248),
    (4, 64, 64, 41, 48, 2): (1, 124672, 25975808, 266496, 99584),
    (4, 64, 64, 41, 64, 2): (1, 124672, 35589120, 349696, 132352),
    (4, 64, 64, 41, 125, 2): (1, 124672, 160965888, 682496, 257280),
    (4, 64, 64, 41, 128, 2): (1, 124672, 169159680, 682496, 263424),
    (4, 64, 64, 48, 1, 2): (1, 207872, 10961920, 16896, 3328),
    (4, 64, 64, 48, 22, 2): (1, 207872, 15203840, 150016, 46336),
    (4, 64, 64, 48, 39, 2): (1, 207872, 21765120, 249856, 81152),
    (4, 64, 64, 48, 40, 2): (1, 207872, 22388224, 249856, 83200),
    (4, 64, 64, 48, 41, 2): (1, 124672, 22731264, 266496, 85248),
    (4, 64, 64, 48, 48, 2): (1, 124672, 28778752, 299776, 99584),
    (4, 64, 64, 48, 64, 2): (1, 124672, 39796224, 399616, 132352),
    (4, 64, 64, 48, 125, 2): (1, 124672, 178608896, 782336, 257280),
    (4, 64, 64, 48, 128, 2): (1, 124672, 187513344, 798976, 263424),
    (4, 64, 64, 64, 1, 2): (1, 207872, 11113984, 16896, 3328),
    (4, 64, 64, 64, 22, 2): (1, 207872, 16984064, 183296, 46336),
    (4, 64, 64, 64, 39, 2): (1, 207872, 26104832, 333056, 81152),
    (4, 64, 64, 64, 40, 2): (1, 207872, 26973184, 333056, 83200),
    (4, 64, 64, 64, 41, 2): (1, 124672, 27407360, 349696, 85248),
    (4, 64, 64, 64, 48, 2): (1, 124672, 35798272, 399616, 99584),
    (4, 64, 64, 64, 64, 2): (1, 124672, 50204160, 532736, 132352),
    (4, 64, 64, 64, 125, 2): (1, 124672, 221957376, 1048576, 257280),
    (4, 64, 64, 64, 128, 2): (1, 124672, 232479232, 1065216, 263424),
    (4, 64, 64, 125, 1, 2): (1, 207872, 11994880, 16896, 3328),
    (4, 64, 64, 125, 22, 2): (1, 207872, 25387008, 366336, 46336),
    (4, 64, 64, 125, 39, 2): (1, 207872, 46556416, 649216, 81152),
    (4, 64, 64, 125, 40, 2): (1, 207872, 48693248, 665856, 83200),
    (4, 64, 64, 125, 41, 2): (1, 124672, 49475328, 682496, 85248),
    (4, 64, 64, 125, 48, 2): (1, 124672, 69778944, 782336, 99584),
    (4, 64, 64, 125, 64, 2): (1, 124672, 99520512, 1048576, 132352),
    (4, 64, 64, 125, 125, 2): (1, 124672, 424766976, 2046976, 257280),
    (4, 64, 64, 125, 128, 2): (1, 124672, 442389504, 2080256, 263424),
    (4, 64, 64, 128, 1, 2): (1, 207872, 12049920, 16896, 3328),
    (4, 64, 64, 128, 22, 2): (1, 207872, 25843200, 366336, 46336),
    (4, 64, 64, 128, 39, 2): (1, 207872, 47690240, 649216, 81152),
    (4, 64, 64, 128, 40, 2): (1, 207872, 49900544, 665856, 83200),
    (4, 64, 64, 128, 41, 2): (1, 124672, 50699264, 682496, 85248),
    (4, 64, 64, 128, 48, 2): (1, 124672, 71740672, 798976, 99584),
    (4, 64, 64, 128, 64, 2): (1, 124672, 102321664, 1065216, 132352),
    (4, 64, 64, 128, 125, 2): (1, 124672, 436244736, 2080256, 257280),
    (4, 64, 64, 128, 128, 2): (1, 124672, 454285824, 2130176, 263424),
}


@pytest.fixture(scope="module")
def lib():
    entry.build()
    return _lib.load_library()


@pytest.mark.parametrize("setting", list(SETTINGS))
def test_dispatch_table(lib, setting, monkeypatch):
    for k in [k for env in SETTINGS.values() for k in env]:
        monkeypatch.delenv(k, raising=False)
    for k, v in SETTINGS[setting].items():
        monkeypatch.setenv(k, v)
    for s in SHAPES:
        n, cin, cout, p, k, nb = s
        got = (lib.dstd_gc_needs_xa(cin, cout, p, k, nb), lib.dstd_gc_fwd_workspace_bytes(n, cin, cout, p, k, nb),
               lib.dstd_gc_bwd_workspace_bytes(n, cin, cout, p, k, nb), lib.dstd_chmix_bwd_workspace_bytes(n, cin, cout, p, k),
               lib.dstd_bn_act_workspace_bytes(n, cout, p, k))
        assert got == TABLE[s], (s, setting)


# ---- GPU: the kernels each DSTD-GC call launches.  A shape or switch that silently fell back to a slower path would
# change these lists while every parity test still passes.
KERNEL_SETTINGS = {**SETTINGS, "agg_gen_mma": {"DSTD_AGG_GEN_MMA": "1"}}
KERNEL_CASES = GC_CASES + STRESS_CASES


def launched_kernels(case):
    """Library kernels launched by one gc_forward + gc_backward, in launch order, names cut at '<' / '(' and
    without the `_kernel` suffix."""
    from torch.profiler import ProfilerActivity, profile
    n, cin, cout, p, k, nb, layout, adj_t, use_skip = case
    g = torch.Generator().manual_seed(3)
    be = gp.cuda_backend()
    x, gout = gp.to_dev(gp.unit_input(g, n, cin, p, k, layout)), gp.to_dev(gp.unit_input(g, n, cout, p, k, layout))
    skip = gp.to_dev(gp.unit_input(g, n, cout, p, k, layout)) if use_skip else None
    alpha = gp.to_dev(gp.rnd((1,), g, 0.3) + 0.5)
    brs = gp.dev_branches(gp.make_branches(g, nb, cin, cout, p, k))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out, m, pd, xa = be.gc_forward(x, alpha, brs, skip, adj_t)
        be.gc_backward(x, gout, alpha, brs, m, pd, xa, adj_t)
        torch.cuda.synchronize()
    evs = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "dstd::" in e.name),
                 key=lambda e: e.time_range.start)
    return " ".join(e.name.removeprefix("void ").removeprefix("dstd::").split("(")[0].split("<")[0].removesuffix("_kernel")
                    for e in evs)


KERNELS = {
    # KERNEL_CASES index: (default switches, {setting: kernels where they differ from the default})
    0: ('pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        {
            'unit_tc': 'pack mproj_fwd dynadj_fwd_mma pack_w16 unit_fwd_tc pack pack_w16 unit_bwd_tc dynadj_bwd_mma mproj_bwd reduce_segments',
            'bf16': 'pack mproj_fwd dynadj_fwd_mma pack_w16 unit_fwd_tc pack pack_w16 unit_bwd_tc dynadj_bwd_mma mproj_bwd reduce_segments',
            'disable_tc': 'pack mproj_fwd dynadj_fwd_mma aggmix_fwd pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        }),
    1: ('pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        {
            'unit_tc': 'pack mproj_fwd dynadj_fwd_mma pack_w16 unit_fwd_tc pack pack_w16 unit_bwd_tc dynadj_bwd_mma mproj_bwd reduce_segments',
            'bf16': 'pack mproj_fwd dynadj_fwd_mma pack_w16 unit_fwd_tc pack pack_w16 unit_bwd_tc dynadj_bwd_mma mproj_bwd reduce_segments',
            'disable_tc': 'pack mproj_fwd dynadj_fwd_mma aggmix_fwd pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        }),
    2: ('pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        {
            'unit_tc': 'pack mproj_fwd dynadj_fwd_mma pack_w16 unit_fwd_tc pack pack_w16 unit_bwd_tc dynadj_bwd_mma mproj_bwd reduce_segments',
            'bf16': 'pack mproj_fwd dynadj_fwd_mma pack_w16 unit_fwd_tc pack pack_w16 unit_bwd_tc dynadj_bwd_mma mproj_bwd reduce_segments',
            'disable_tc': 'pack mproj_fwd dynadj_fwd_mma aggmix_fwd pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        }),
    3: ('pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        {
            'unit_tc': 'pack mproj_fwd dynadj_fwd_mma pack_w16 unit_fwd_tc pack pack_w16 unit_bwd_tc dynadj_bwd_mma mproj_bwd reduce_segments',
            'bf16': 'pack mproj_fwd dynadj_fwd_mma pack_w16 unit_fwd_tc pack pack_w16 unit_bwd_tc dynadj_bwd_mma mproj_bwd reduce_segments',
            'disable_tc': 'pack mproj_fwd dynadj_fwd_mma aggmix_fwd pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        }),
    4: ('pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        {
            'unit_tc': 'pack mproj_fwd dynadj_fwd_mma pack_w16 unit_fwd_tc pack pack_w16 unit_bwd_tc dynadj_bwd_mma mproj_bwd reduce_segments',
            'bf16': 'pack mproj_fwd dynadj_fwd_mma pack_w16 unit_fwd_tc pack pack_w16 unit_bwd_tc dynadj_bwd_mma mproj_bwd reduce_segments',
            'disable_tc': 'pack mproj_fwd dynadj_fwd_mma aggmix_fwd pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        }),
    5: ('pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        {
            'unit_tc': 'pack mproj_fwd dynadj_fwd_mma pack_w16 unit_fwd_tc pack pack_w16 unit_bwd_tc dynadj_bwd_mma mproj_bwd reduce_segments',
            'bf16': 'pack mproj_fwd dynadj_fwd_mma pack_w16 unit_fwd_tc pack pack_w16 unit_bwd_tc dynadj_bwd_mma mproj_bwd reduce_segments',
            'disable_tc': 'pack mproj_fwd dynadj_fwd_mma aggmix_fwd pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        }),
    6: ('pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        {
            'unit_tc': 'pack mproj_fwd dynadj_fwd_mma pack_w16 unit_fwd_tc pack pack_w16 unit_bwd_tc dynadj_bwd_mma mproj_bwd reduce_segments',
            'bf16': 'pack mproj_fwd dynadj_fwd_mma pack_w16 unit_fwd_tc pack pack_w16 unit_bwd_tc dynadj_bwd_mma mproj_bwd reduce_segments',
            'disable_tc': 'pack mproj_fwd dynadj_fwd_mma aggmix_fwd pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        }),
    7: ('pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        {
            'unit_tc': 'pack mproj_fwd dynadj_fwd_mma pack_w16 unit_fwd_tc pack pack_w16 unit_bwd_tc dynadj_bwd_mma mproj_bwd reduce_segments',
            'bf16': 'pack mproj_fwd dynadj_fwd_mma pack_w16 unit_fwd_tc pack pack_w16 unit_bwd_tc dynadj_bwd_mma mproj_bwd reduce_segments',
            'disable_tc': 'pack mproj_fwd dynadj_fwd_mma aggmix_fwd pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        }),
    8: ('pack mproj_fwd dynadj_fwd_mma pack_tc aggmix_fwd_tc pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        {
            'unit_tc': 'pack mproj_fwd dynadj_fwd_mma pack_w16 unit_fwd_tc pack pack_w16 unit_bwd_tc dynadj_bwd_mma mproj_bwd reduce_segments',
            'bf16': 'pack mproj_fwd dynadj_fwd_mma pack_w16 unit_fwd_tc pack pack_w16 unit_bwd_tc dynadj_bwd_mma mproj_bwd reduce_segments',
            'disable_tc': 'pack mproj_fwd dynadj_fwd_mma aggmix_fwd pack aggmix_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        }),
    9: ('pack mproj_fwd dynadj_fwd_gen aggregate_fwd_gen bgemm pack bgemm wgrad aggregate_bwd_gen dynadj_bwd_gen gm2_reduce mproj_bwd reduce_segments', {}),
    10: ('pack mproj_fwd dynadj_fwd_gen aggregate_fwd_gen bgemm pack bgemm wgrad aggregate_bwd_gen dynadj_bwd_gen gm2_reduce mproj_bwd reduce_segments',
        {
            'agg_gen_mma': 'pack mproj_fwd dynadj_fwd_gen aggregate_fwd_gen_mma bgemm pack bgemm wgrad aggregate_bwd_gen dynadj_bwd_gen gm2_reduce mproj_bwd reduce_segments',
        }),
    11: ('pack mproj_fwd dynadj_fwd_gen aggregate_fwd_gen bgemm bgemm pack bgemm_tc_pack bgemm_tc wgrad aggregate_bwd_gen dynadj_bwd_gen gm2_reduce mproj_bwd reduce_segments',
        {
            'bgemm_cuda_core': 'pack mproj_fwd dynadj_fwd_gen aggregate_fwd_gen bgemm bgemm pack bgemm wgrad aggregate_bwd_gen dynadj_bwd_gen gm2_reduce mproj_bwd reduce_segments',
        }),
    12: ('pack mproj_fwd dynadj_fwd_gen aggregate_fwd_gen bgemm pack bgemm wgrad aggregate_bwd_gen dynadj_bwd_gen gm2_reduce mproj_bwd reduce_segments',
        {
            'agg_gen_mma': 'pack mproj_fwd dynadj_fwd_gen aggregate_fwd_gen_mma bgemm pack bgemm wgrad aggregate_bwd_gen dynadj_bwd_gen gm2_reduce mproj_bwd reduce_segments',
        }),
    13: ('pack mproj_fwd dynadj_fwd_mma aggmix_fwd pack bgemm_tc_pack bgemm_tc wgrad_tc aggregate_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        {
            'bgemm_cuda_core': 'pack mproj_fwd dynadj_fwd_mma aggmix_fwd pack bgemm bgemm wgrad aggregate_bwd dynadj_bwd_mma mproj_bwd reduce_segments',
        }),
    14: ('pack mproj_fwd dynadj_fwd_gen aggregate_fwd_gen bgemm_tc_pack bgemm_tc pack bgemm_tc_pack bgemm_tc wgrad_tc aggregate_bwd_gen dynadj_bwd_gen gm2_reduce bgemm wgrad reduce_segments',
        {
            'bgemm_cuda_core': 'pack mproj_fwd dynadj_fwd_gen aggregate_fwd_gen bgemm pack bgemm bgemm wgrad aggregate_bwd_gen dynadj_bwd_gen gm2_reduce bgemm wgrad reduce_segments',
        }),
    15: ('pack mproj_fwd dynadj_fwd_gen aggregate_fwd_gen bgemm_tc_pack bgemm_tc pack bgemm_tc_pack bgemm_tc wgrad_tc aggregate_bwd_gen dynadj_bwd_gen gm2_reduce bgemm wgrad reduce_segments',
        {
            'bgemm_cuda_core': 'pack mproj_fwd dynadj_fwd_gen aggregate_fwd_gen bgemm pack bgemm bgemm wgrad aggregate_bwd_gen dynadj_bwd_gen gm2_reduce bgemm wgrad reduce_segments',
            'agg_gen_mma': 'pack mproj_fwd dynadj_fwd_gen aggregate_fwd_gen_mma bgemm_tc_pack bgemm_tc pack bgemm_tc_pack bgemm_tc wgrad_tc aggregate_bwd_gen dynadj_bwd_gen gm2_reduce bgemm wgrad reduce_segments',
        }),
}


@pytest.mark.gpu
@pytest.mark.parametrize("setting", list(KERNEL_SETTINGS))
def test_kernel_paths(setting, monkeypatch):
    for k in [k for env in KERNEL_SETTINGS.values() for k in env]:
        monkeypatch.delenv(k, raising=False)
    for k, v in KERNEL_SETTINGS[setting].items():
        monkeypatch.setenv(k, v)
    for i, case in enumerate(KERNEL_CASES):
        dflt, over = KERNELS[i]
        assert launched_kernels(case) == over.get(setting, dflt), (case, setting)


# ---- GPU: the BatchNorm kernels each bn_act call launches, with their template arguments and launch geometry.  The
# parity tests pass whichever compiled U or twin a dispatch picks; this table does not.
def _bn_cases():
    from tests import test_custom_skeleton as cs
    cases = {}
    for src, rows, full in (("parity", gp.BN_CASES, True), ("parity_fast", gp.BN_FAST_CASES, False),
                            ("skeleton", cs.BN_CASES, True), ("skeleton_fast", cs.BN_FAST_CASES, False)):
        for i, row in enumerate(rows):
            if not full:   # n, c, t, v, y_order, r_order, out_order, prelu, training -> the full form
                n, c, t, v, yo, ro, oo, use_prelu, training = row
                row = (n, c, t, v, yo, ro, oo, False, use_prelu, False, training)
            cases[f"{src}/{i}"] = row
    return cases


BN_CASES = _bn_cases()
BN_SYNC_CASES = ("parity/0", "skeleton/2")   # generic and fast (DSTD_BN_FAST=0 / 1), V <= 32 and V > 32


def _bn_launch_log(fn):
    """Library kernels `fn` launches, in order: 'name<template args> grid block smem', names without 'dstd::'."""
    import json
    import tempfile
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = f"{d}/trace.json"
        prof.export_chrome_trace(path)
        with open(path) as f:
            evs = json.load(f)["traceEvents"]
    evs = sorted((e for e in evs if e.get("cat") == "kernel" and "dstd::" in e["name"]), key=lambda e: e["ts"])
    out = []
    for e in evs:
        a = e.get("args", {})
        geom = "x".join(map(str, a.get("grid", ()))), "x".join(map(str, a.get("block", ()))), a.get("shared memory")
        out.append(e["name"].removeprefix("void ").removeprefix("dstd::").split("(")[0] + " %s %s %s" % geom)
    return out


def _bn_inputs(case):
    from dstd_gcn_b200.ops import _out_like
    n, c, t, v, yo, ro, out_order, vc, use_prelu, use_mask, training = case
    g = torch.Generator().manual_seed(n * 13 + c + v)
    d = dict(y=gp.to_dev(gp._ordered(g, n, c, t, v, yo) * 2.0 + 3.0),
             r=gp.to_dev(gp._ordered(g, n, c, t, v, ro)) if ro else None,
             gamma=gp.to_dev(gp.rnd((c * v,), g, 0.5) + 1.0), beta=gp.to_dev(gp.rnd((c * v,), g, 0.5)),
             rm=torch.zeros(c * v, device=gp.DEV), rv=torch.ones(c * v, device=gp.DEV),
             nbt=torch.zeros((), dtype=torch.int64, device=gp.DEV),
             prelu=gp.to_dev(torch.tensor([0.25], dtype=torch.float64)) if use_prelu else None,
             mask=gp.to_dev((torch.rand((n, c, t, v), generator=g) > 0.1).double() / 0.9) if use_mask else None)
    d["out_like"] = _out_like(d["y"], out_order) if out_order else None
    return d


def bn_launches(case):
    """Kernels of one forward, one backward and, with a residual, one backward with gr_add."""
    n, c, t, v, yo, ro, out_order, vc, use_prelu, use_mask, training = case
    be, d = gp.cuda_backend(), _bn_inputs(case)
    y, r, prelu, mask = d["y"], d["r"], d["prelu"], d["mask"]
    fwd = lambda: be.bn_act_forward(y, r, d["gamma"], d["beta"], d["rm"], d["rv"], d["nbt"] if training else None,
                                    prelu, mask, vc, training, 1e-5, 0.1, d["out_like"])
    out, mean, istd = fwd()
    gout = torch.randn_like(out)
    bwd = lambda gadd=None: be.bn_act_backward(y, r, gout, d["gamma"], d["beta"], prelu, mask, mean, istd, vc,
                                               training, r is not None, gadd)
    log = {"fwd": _bn_launch_log(fwd), "bwd": _bn_launch_log(bwd)}
    if r is not None:
        gadd = torch.randn_like(out)
        log["bwd_add"] = _bn_launch_log(lambda: bwd(gadd))
    return log


def bn_sync_launches(case):
    """Kernels of the four phases of a synchronised BN call on one rank."""
    n, c, t, v, yo, ro, out_order, vc, use_prelu, use_mask, training = case
    be, d = gp.cuda_backend(), _bn_inputs(case)
    y, r, prelu, mask = d["y"], d["r"], d["prelu"], d["mask"]
    res = {}
    log = {"fwd_local": _bn_launch_log(lambda: res.update(rows=be.bn_act_forward_local(y, vc)))}
    log["fwd_global"] = _bn_launch_log(lambda: res.update(fwd=be.bn_act_forward_global(
        y, r, d["gamma"], d["beta"], d["rm"], d["rv"], d["nbt"], prelu, mask, vc, 1e-5, 0.1, res["rows"],
        d["out_like"])))
    out, mean, istd = res["fwd"]
    gout = torch.randn_like(out)
    log["bwd_local"] = _bn_launch_log(lambda: res.update(bwd=be.bn_act_backward_local(
        y, r, gout, d["gamma"], d["beta"], prelu, mask, mean, istd, vc, r is not None)))
    rows, gy, gr = res["bwd"][3:]
    log["bwd_global"] = _bn_launch_log(lambda: be.bn_act_backward_global(
        y, r, gout, d["gamma"], d["beta"], prelu, mask, mean, istd, vc, rows, gy, gr))
    return log


REFUSED = "refused"   # T*V above the generic kernels' limit with the fast path off: the call raises

# case id (BN_CASES, or sync/<id> of BN_SYNC_CASES): {'1': the launches of each call with DSTD_BN_FAST=1, '0': the
# same with DSTD_BN_FAST=0 where they differ}.  A launch: 'kernel<template args> grid block shared-memory-bytes' (static
# + dynamic, as the profiler reports it).
BN_LAUNCHES = {
    'parity/0': {
        '1': {
            'fwd': [
                'bn_stats_kernel<2> 16x1x1 416x1x1 6160',
                'bnf_apply_kernel<4, 4, true, false> 8x1x1 416x1x1 101136',
            ],
            'bwd': [
                'bnf_bwd_reduce_kernel<4, 2, true, false> 8x1x1 416x1x1 76112',
                'bnf_bwd_apply_kernel<4, 2, true, true, false, false> 8x1x1 416x1x1 78672',
            ],
            'bwd_add': [
                'bnf_bwd_reduce_kernel<4, 2, true, false> 8x1x1 416x1x1 76112',
                'bnf_bwd_apply_kernel<4, 2, true, true, true, false> 8x1x1 416x1x1 103312',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<2> 16x1x1 416x1x1 6160',
                'bn_apply_kernel<2, 4> 16x1x1 416x1x1 50048',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<2, 4> 16x1x1 416x1x1 74048',
                'bn_bwd_apply_kernel<2, 4> 16x1x1 416x1x1 86880',
            ],
            'bwd_add': [
                'bn_bwd_reduce_kernel<2, 4> 16x1x1 416x1x1 74048',
                'bn_bwd_apply_add_kernel<2, 4> 16x1x1 416x1x1 111520',
            ],
        },
    },
    'parity/1': {
        '1': {
            'fwd': [
                'bn_stats_kernel<2> 16x1x1 416x1x1 6160',
                'bn_apply_kernel<2, 4> 16x1x1 416x1x1 25408',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<2, 4> 16x1x1 416x1x1 49408',
                'bn_bwd_apply_kernel<2, 4> 16x1x1 416x1x1 62240',
            ],
        },
    },
    'parity/2': {
        '1': {
            'fwd': [
                'bn_stats_kernel<1> 8x1x1 256x1x1 2000',
                'bnf_apply_kernel<4, 4, false, false> 4x1x1 128x1x1 18576',
            ],
            'bwd': [
                'bnf_bwd_reduce_kernel<4, 4, false, false> 4x1x1 128x1x1 34192',
                'bnf_bwd_apply_kernel<4, 4, false, false, false, false> 4x1x1 128x1x1 36752',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<1> 8x1x1 256x1x1 2000',
                'bn_apply_kernel<1, 4> 8x1x1 256x1x1 8768',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<1, 4> 8x1x1 256x1x1 16128',
                'bn_bwd_apply_kernel<1, 4> 8x1x1 256x1x1 20640',
            ],
        },
    },
    'parity/3': {
        '1': {
            'fwd': [
                'bn_eval_stats_kernel 2x1x1 128x1x1 0',
                'bnf_apply_kernel<4, 4, true, false> 8x1x1 256x1x1 61456',
            ],
            'bwd': [
                'bnf_bwd_reduce_kernel<4, 4, true, false> 8x1x1 256x1x1 90512',
                'bnf_bwd_apply_kernel<4, 4, true, true, false, false> 8x1x1 256x1x1 93072',
            ],
            'bwd_add': [
                'bnf_bwd_reduce_kernel<4, 4, true, false> 8x1x1 256x1x1 90512',
                'bnf_bwd_apply_kernel<4, 2, true, true, true, false> 8x1x1 256x1x1 63632',
            ],
        },
        '0': {
            'fwd': [
                'bn_eval_stats_kernel 2x1x1 128x1x1 0',
                'bn_apply_kernel<2, 4> 8x1x1 480x1x1 59648',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<2, 4> 8x1x1 480x1x1 88448',
                'bn_bwd_apply_kernel<2, 4> 8x1x1 480x1x1 103680',
            ],
            'bwd_add': [
                'bn_bwd_reduce_kernel<2, 4> 8x1x1 480x1x1 88448',
                'bn_bwd_apply_add_kernel<2, 2> 8x1x1 480x1x1 66880',
            ],
        },
    },
    'parity/4': {
        '1': {
            'fwd': [
                'bn_stats_kernel<2> 64x2x1 416x1x1 6160',
                'bnf_apply_kernel<4, 4, false, false> 32x2x1 416x1x1 51856',
            ],
            'bwd': [
                'bnf_bwd_reduce_kernel<4, 4, false, false> 32x2x1 416x1x1 100752',
                'bnf_bwd_apply_kernel<4, 4, false, false, false, false> 32x2x1 416x1x1 103312',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<2> 64x2x1 416x1x1 6160',
                'bn_apply_kernel<2, 4> 64x2x1 416x1x1 25408',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<2, 4> 64x2x1 416x1x1 49408',
                'bn_bwd_apply_kernel<2, 4> 64x2x1 416x1x1 62240',
            ],
        },
    },
    'parity/5': {
        '1': {
            'fwd': [
                'bn_stats_kernel<2> 3x1x1 416x1x1 6160',
                'bn_apply_kernel<2, 4> 3x1x1 416x1x1 50048',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<2, 4> 3x1x1 416x1x1 74048',
                'bn_bwd_apply_kernel<2, 4> 3x1x1 416x1x1 86880',
            ],
            'bwd_add': [
                'bn_bwd_reduce_kernel<2, 4> 3x1x1 416x1x1 74048',
                'bn_bwd_apply_add_kernel<2, 4> 3x1x1 416x1x1 111520',
            ],
        },
    },
    'parity_fast/0': {
        '1': {
            'fwd': [
                'bn_stats_kernel<2> 8x2x1 416x1x1 6160',
                'bnf_apply_kernel<4, 4, true, false> 4x2x1 416x1x1 101136',
            ],
            'bwd': [
                'bnf_bwd_reduce_kernel<4, 2, true, false> 4x2x1 416x1x1 76112',
                'bnf_bwd_apply_kernel<4, 2, true, true, false, false> 4x2x1 416x1x1 78672',
            ],
            'bwd_add': [
                'bnf_bwd_reduce_kernel<4, 2, true, false> 4x2x1 416x1x1 76112',
                'bnf_bwd_apply_kernel<4, 2, true, true, true, false> 4x2x1 416x1x1 103312',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<2> 8x2x1 416x1x1 6160',
                'bn_apply_kernel<2, 4> 8x2x1 416x1x1 50048',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<2, 4> 8x2x1 416x1x1 74048',
                'bn_bwd_apply_kernel<2, 4> 8x2x1 416x1x1 86880',
            ],
            'bwd_add': [
                'bn_bwd_reduce_kernel<2, 4> 8x2x1 416x1x1 74048',
                'bn_bwd_apply_add_kernel<2, 4> 8x2x1 416x1x1 111520',
            ],
        },
    },
    'parity_fast/1': {
        '1': {
            'fwd': [
                'bn_stats_kernel<2> 8x1x1 416x1x1 6160',
                'bnf_apply_kernel<4, 4, false, false> 4x1x1 416x1x1 51856',
            ],
            'bwd': [
                'bnf_bwd_reduce_kernel<4, 4, false, false> 4x1x1 416x1x1 100752',
                'bnf_bwd_apply_kernel<4, 4, false, false, false, false> 4x1x1 416x1x1 103312',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<2> 8x1x1 416x1x1 6160',
                'bn_apply_kernel<2, 4> 8x1x1 416x1x1 25408',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<2, 4> 8x1x1 416x1x1 49408',
                'bn_bwd_apply_kernel<2, 4> 8x1x1 416x1x1 62240',
            ],
        },
    },
    'parity_fast/2': {
        '1': {
            'fwd': [
                'bn_stats_kernel<2> 4x1x1 480x1x1 7360',
                'bnf_apply_kernel<4, 4, true, false> 4x1x1 256x1x1 61456',
            ],
            'bwd': [
                'bnf_bwd_reduce_kernel<4, 4, true, false> 4x1x1 256x1x1 90512',
                'bnf_bwd_apply_kernel<4, 4, true, true, false, false> 4x1x1 256x1x1 93072',
            ],
            'bwd_add': [
                'bnf_bwd_reduce_kernel<4, 4, true, false> 4x1x1 256x1x1 90512',
                'bnf_bwd_apply_kernel<4, 2, true, true, true, false> 4x1x1 256x1x1 63632',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<2> 4x1x1 480x1x1 7360',
                'bn_apply_kernel<2, 4> 4x1x1 480x1x1 59648',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<2, 4> 4x1x1 480x1x1 88448',
                'bn_bwd_apply_kernel<2, 4> 4x1x1 480x1x1 103680',
            ],
            'bwd_add': [
                'bn_bwd_reduce_kernel<2, 4> 4x1x1 480x1x1 88448',
                'bn_bwd_apply_add_kernel<2, 2> 4x1x1 480x1x1 66880',
            ],
        },
    },
    'parity_fast/3': {
        '1': {
            'fwd': [
                'bn_stats_kernel<2> 8x1x1 448x1x1 7000',
                'bnf_apply_kernel<8, 2, true, false> 2x1x1 448x1x1 114576',
            ],
            'bwd': [
                'bnf_bwd_reduce_kernel<8, 1, true, false> 2x1x1 448x1x1 86192',
                'bnf_bwd_apply_kernel<8, 1, true, true, false, false> 2x1x1 448x1x1 88752',
            ],
            'bwd_add': [
                'bnf_bwd_reduce_kernel<8, 1, true, false> 2x1x1 448x1x1 86192',
                'bnf_bwd_apply_kernel<8, 1, true, true, true, false> 2x1x1 448x1x1 116752',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<2> 8x1x1 448x1x1 7000',
                'bn_apply_kernel<2, 4> 8x1x1 448x1x1 56768',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<2, 4> 8x1x1 448x1x1 84128',
                'bn_bwd_apply_kernel<2, 4> 8x1x1 448x1x1 98640',
            ],
            'bwd_add': [
                'bn_bwd_reduce_kernel<2, 4> 8x1x1 448x1x1 84128',
                'bn_bwd_apply_add_kernel<2, 2> 8x1x1 448x1x1 63640',
            ],
        },
    },
    'parity_fast/4': {
        '1': {
            'fwd': [
                'bn_eval_stats_kernel 2x1x1 128x1x1 0',
                'bnf_apply_kernel<8, 4, false, false> 2x1x1 448x1x1 114576',
            ],
            'bwd': [
                'bnf_bwd_reduce_kernel<8, 2, false, false> 2x1x1 448x1x1 114192',
                'bnf_bwd_apply_kernel<8, 2, false, false, false, false> 2x1x1 448x1x1 116752',
            ],
        },
        '0': {
            'fwd': [
                'bn_eval_stats_kernel 2x1x1 128x1x1 0',
                'bn_apply_kernel<2, 4> 8x1x1 448x1x1 28768',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<2, 4> 8x1x1 448x1x1 56128',
                'bn_bwd_apply_kernel<2, 4> 8x1x1 448x1x1 70640',
            ],
        },
    },
    'parity_fast/5': {
        '1': {
            'fwd': [
                'bn_stats_kernel<1> 4x1x1 224x1x1 1760',
                'bnf_apply_kernel<4, 4, false, false> 4x1x1 64x1x1 9616',
            ],
            'bwd': [
                'bnf_bwd_reduce_kernel<4, 4, false, false> 4x1x1 64x1x1 16272',
                'bnf_bwd_apply_kernel<4, 4, false, false, false, false> 4x1x1 64x1x1 18832',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<1> 4x1x1 224x1x1 1760',
                'bn_apply_kernel<1, 4> 4x1x1 224x1x1 7808',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<1, 4> 4x1x1 224x1x1 14208',
                'bn_bwd_apply_kernel<1, 4> 4x1x1 224x1x1 18240',
            ],
        },
    },
    'parity_fast/6': {
        '1': {
            'fwd': [
                'bn_stats_kernel<8> 4x1x1 352x1x1 22000',
                'bnf_apply_kernel<8, 2, true, true> 2x1x1 704x1x1 178576',
            ],
            'bwd': [
                'bnf_bwd_reduce_kernel<8, 1, true, true> 2x1x1 704x1x1 134192',
                'bnf_bwd_apply_kernel<8, 1, true, true, false, true> 2x1x1 704x1x1 136752',
            ],
            'bwd_add': [
                'bnf_bwd_reduce_kernel<8, 1, true, true> 2x1x1 704x1x1 134192',
                'bnf_bwd_apply_kernel<8, 1, true, true, true, true> 2x1x1 704x1x1 180752',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<8> 4x1x1 352x1x1 22000',
                'bn_apply_kernel<8, 2> 4x1x1 352x1x1 88768',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<8, 1> 4x1x1 352x1x1 66128',
                'bn_bwd_apply_kernel<8, 1> 4x1x1 352x1x1 77640',
            ],
            'bwd_add': [
                'bn_bwd_reduce_kernel<8, 1> 4x1x1 352x1x1 66128',
                'bn_bwd_apply_add_kernel<8, 1> 4x1x1 352x1x1 99640',
            ],
        },
    },
    'parity_fast/7': {
        '1': {
            'fwd': [
                'bn_stats_kernel<8> 4x1x1 352x1x1 22000',
                'bnf_apply_kernel<8, 2, false, true> 2x1x1 704x1x1 90576',
            ],
            'bwd': [
                'bnf_bwd_reduce_kernel<8, 2, false, true> 2x1x1 704x1x1 178192',
                'bnf_bwd_apply_kernel<8, 2, false, false, false, true> 2x1x1 704x1x1 180752',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<8> 4x1x1 352x1x1 22000',
                'bn_apply_kernel<8, 4> 4x1x1 352x1x1 88768',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<8, 2> 4x1x1 352x1x1 88128',
                'bn_bwd_apply_kernel<8, 2> 4x1x1 352x1x1 110640',
            ],
        },
    },
    'skeleton/0': {
        '1': {
            'fwd': [
                'bn_stats_kernel<4> 8x1x1 320x1x1 9240',
                'bn_apply_wide_kernel<4, 4> 8x1x1 320x1x1 76992',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<4, 2> 8x1x1 320x1x1 55568',
                'bn_bwd_apply_wide_kernel<4, 2> 8x1x1 320x1x1 66856',
            ],
            'bwd_add': [
                'bn_bwd_reduce_kernel<4, 2> 8x1x1 320x1x1 55568',
                'bn_bwd_apply_add_wide_kernel<4, 2> 8x1x1 320x1x1 85336',
            ],
        },
    },
    'skeleton/1': {
        '1': {
            'fwd': [
                'bn_stats_kernel<4> 8x1x1 352x1x1 10640',
                'bn_apply_wide_kernel<4, 4> 8x1x1 352x1x1 45632',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<4, 4> 8x1x1 352x1x1 85248',
                'bn_bwd_apply_wide_kernel<4, 4> 8x1x1 352x1x1 108576',
            ],
        },
    },
    'skeleton/2': {
        '1': {
            'fwd': [
                'bn_stats_kernel<4> 8x1x1 352x1x1 10640',
                'bnf_apply_wide_kernel<8, 2, true, false> 4x1x1 352x1x1 95376',
            ],
            'bwd': [
                'bnf_bwd_reduce_wide_kernel<8, 1, true, false> 4x1x1 352x1x1 72176',
                'bnf_bwd_apply_wide_kernel<8, 1, true, true, false, false> 4x1x1 352x1x1 82416',
            ],
            'bwd_add': [
                'bnf_bwd_reduce_wide_kernel<8, 1, true, false> 4x1x1 352x1x1 72176',
                'bnf_bwd_apply_wide_kernel<8, 1, true, true, true, false> 4x1x1 352x1x1 103696',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<4> 8x1x1 352x1x1 10640',
                'bn_apply_wide_kernel<4, 4> 8x1x1 352x1x1 88192',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<4, 2> 8x1x1 352x1x1 63968',
                'bn_bwd_apply_wide_kernel<4, 2> 8x1x1 352x1x1 76656',
            ],
            'bwd_add': [
                'bn_bwd_reduce_kernel<4, 2> 8x1x1 352x1x1 63968',
                'bn_bwd_apply_add_wide_kernel<4, 2> 8x1x1 352x1x1 97936',
            ],
        },
    },
    'skeleton/3': {
        '1': {
            'fwd': [
                'bn_stats_kernel<4> 16x2x1 352x1x1 10640',
                'bnf_apply_wide_kernel<8, 4, false, false> 8x2x1 352x1x1 95376',
            ],
            'bwd': [
                'bnf_bwd_reduce_wide_kernel<8, 2, false, false> 8x2x1 352x1x1 93456',
                'bnf_bwd_apply_wide_kernel<8, 2, false, false, false, false> 8x2x1 352x1x1 103696',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<4> 16x2x1 352x1x1 10640',
                'bn_apply_wide_kernel<4, 4> 16x2x1 352x1x1 45632',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<4, 4> 16x2x1 352x1x1 85248',
                'bn_bwd_apply_wide_kernel<4, 4> 16x2x1 352x1x1 108576',
            ],
        },
    },
    'skeleton/4': {
        '1': {
            'fwd': [
                'bn_eval_stats_kernel 4x1x1 128x1x1 0',
                'bn_apply_wide_kernel<4, 2> 8x1x1 512x1x1 64672',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<4, 2> 8x1x1 512x1x1 92528',
                'bn_bwd_apply_wide_kernel<4, 2> 8x1x1 512x1x1 109976',
            ],
            'bwd_add': [
                'bn_bwd_reduce_kernel<4, 2> 8x1x1 512x1x1 92528',
                'bn_bwd_apply_add_wide_kernel<4, 1> 8x1x1 512x1x1 71476',
            ],
        },
    },
    'skeleton/5': {
        '1': {
            'fwd': [
                'bn_stats_kernel<8> 4x1x1 288x1x1 17920',
                'bnf_apply_wide_kernel<8, 2, true, false> 4x1x1 288x1x1 81936',
            ],
            'bwd': [
                'bnf_bwd_reduce_wide_kernel<8, 1, true, false> 4x1x1 288x1x1 62096',
                'bnf_bwd_apply_wide_kernel<8, 1, true, true, false, false> 4x1x1 288x1x1 72336',
            ],
            'bwd_add': [
                'bnf_bwd_reduce_wide_kernel<8, 1, true, false> 4x1x1 288x1x1 62096',
                'bnf_bwd_apply_wide_kernel<8, 1, true, true, true, false> 4x1x1 288x1x1 90256',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<8> 4x1x1 288x1x1 17920',
                'bn_apply_wide_kernel<8, 2> 4x1x1 288x1x1 74752',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<8, 1> 4x1x1 288x1x1 53888',
                'bn_bwd_apply_wide_kernel<8, 1> 4x1x1 288x1x1 64896',
            ],
            'bwd_add': [
                'bn_bwd_reduce_kernel<8, 1> 4x1x1 288x1x1 53888',
                'bn_bwd_apply_add_wide_kernel<8, 1> 4x1x1 288x1x1 82816',
            ],
        },
    },
    'skeleton/6': {
        '1': {
            'fwd': [
                'bn_eval_stats_kernel 2x1x1 128x1x1 0',
                'bnf_apply_wide_kernel<8, 4, false, false> 4x1x1 288x1x1 81936',
            ],
            'bwd': [
                'bnf_bwd_reduce_wide_kernel<8, 2, false, false> 4x1x1 288x1x1 80016',
                'bnf_bwd_apply_wide_kernel<8, 2, false, false, false, false> 4x1x1 288x1x1 90256',
            ],
        },
        '0': {
            'fwd': [
                'bn_eval_stats_kernel 2x1x1 128x1x1 0',
                'bn_apply_wide_kernel<8, 4> 4x1x1 288x1x1 74752',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<8, 2> 4x1x1 288x1x1 71808',
                'bn_bwd_apply_wide_kernel<8, 2> 4x1x1 288x1x1 91776',
            ],
        },
    },
    'skeleton/7': {
        '1': {
            'fwd': [
                'bn_stats_big_kernel 4x1x1 576x1x1 35840',
                'bnf_apply_wide_kernel<8, 2, true, true> 4x1x1 576x1x1 153616',
            ],
            'bwd': [
                'bnf_bwd_reduce_wide_kernel<8, 1, true, true> 4x1x1 576x1x1 115856',
                'bnf_bwd_apply_wide_kernel<8, 1, true, true, false, true> 4x1x1 576x1x1 126096',
            ],
            'bwd_add': [
                'bnf_bwd_reduce_wide_kernel<8, 1, true, true> 4x1x1 576x1x1 115856',
                'bnf_bwd_apply_wide_kernel<8, 1, true, true, true, true> 4x1x1 576x1x1 161936',
            ],
        },
        '0': REFUSED,
    },
    'skeleton/8': {
        '1': {
            'fwd': [
                'bn_stats_kernel<8> 4x1x1 512x1x1 32768',
                'bn_apply_wide_kernel<8, 2> 4x1x1 512x1x1 68608',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<8, 1> 4x1x1 512x1x1 65664',
                'bn_bwd_apply_wide_kernel<8, 1> 4x1x1 512x1x1 84096',
            ],
        },
    },
    'skeleton/9': {
        '1': {
            'fwd': [
                'bn_eval_stats_kernel 4x1x1 128x1x1 0',
                'bnf_apply_wide_kernel<8, 1, true, false> 4x1x1 512x1x1 75792',
            ],
            'bwd': [
                'bnf_bwd_reduce_wide_kernel<8, 1, true, false> 4x1x1 512x1x1 106640',
                'bnf_bwd_apply_wide_kernel<8, 1, true, true, false, false> 4x1x1 512x1x1 116880',
            ],
            'bwd_add': [
                'bn_bwd_reduce_kernel<8, 1> 4x1x1 512x1x1 98432',
                'bn_bwd_apply_add_wide_kernel<8, 1> 4x1x1 512x1x1 149632',
            ],
        },
        '0': {
            'fwd': [
                'bn_eval_stats_kernel 4x1x1 128x1x1 0',
                'bn_apply_wide_kernel<8, 1> 4x1x1 512x1x1 68608',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<8, 1> 4x1x1 512x1x1 98432',
                'bn_bwd_apply_wide_kernel<8, 1> 4x1x1 512x1x1 116864',
            ],
            'bwd_add': [
                'bn_bwd_reduce_kernel<8, 1> 4x1x1 512x1x1 98432',
                'bn_bwd_apply_add_wide_kernel<8, 1> 4x1x1 512x1x1 149632',
            ],
        },
    },
    'skeleton/10': {
        '1': {
            'fwd': [
                'bn_stats_kernel<1> 3x1x1 224x1x1 1600',
                'bnf_apply_wide_kernel<4, 4, true, false> 3x1x1 128x1x1 23056',
            ],
            'bwd': [
                'bnf_bwd_reduce_wide_kernel<4, 4, true, false> 3x1x1 128x1x1 27536',
                'bnf_bwd_apply_wide_kernel<4, 4, true, true, false, false> 3x1x1 128x1x1 37776',
            ],
            'bwd_add': [
                'bnf_bwd_reduce_wide_kernel<4, 4, true, false> 3x1x1 128x1x1 27536',
                'bnf_bwd_apply_wide_kernel<4, 4, true, true, true, false> 3x1x1 128x1x1 44176',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<1> 3x1x1 224x1x1 1600',
                'bn_apply_wide_kernel<1, 4> 3x1x1 224x1x1 15872',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<1, 4> 3x1x1 224x1x1 19328',
                'bn_bwd_apply_wide_kernel<1, 4> 3x1x1 224x1x1 24576',
            ],
            'bwd_add': [
                'bn_bwd_reduce_kernel<1, 4> 3x1x1 224x1x1 19328',
                'bn_bwd_apply_add_wide_kernel<1, 4> 3x1x1 224x1x1 30976',
            ],
        },
    },
    'skeleton_fast/0': {
        '1': {
            'fwd': [
                'bn_stats_kernel<4> 8x2x1 352x1x1 10640',
                'bnf_apply_wide_kernel<8, 2, true, false> 4x2x1 352x1x1 95376',
            ],
            'bwd': [
                'bnf_bwd_reduce_wide_kernel<8, 1, true, false> 4x2x1 352x1x1 72176',
                'bnf_bwd_apply_wide_kernel<8, 1, true, true, false, false> 4x2x1 352x1x1 82416',
            ],
            'bwd_add': [
                'bnf_bwd_reduce_wide_kernel<8, 1, true, false> 4x2x1 352x1x1 72176',
                'bnf_bwd_apply_wide_kernel<8, 1, true, true, true, false> 4x2x1 352x1x1 103696',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<4> 8x2x1 352x1x1 10640',
                'bn_apply_wide_kernel<4, 4> 8x2x1 352x1x1 88192',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<4, 2> 8x2x1 352x1x1 63968',
                'bn_bwd_apply_wide_kernel<4, 2> 8x2x1 352x1x1 76656',
            ],
            'bwd_add': [
                'bn_bwd_reduce_kernel<4, 2> 8x2x1 352x1x1 63968',
                'bn_bwd_apply_add_wide_kernel<4, 2> 8x2x1 352x1x1 97936',
            ],
        },
    },
    'skeleton_fast/1': {
        '1': {
            'fwd': [
                'bn_stats_kernel<4> 8x1x1 352x1x1 10640',
                'bnf_apply_wide_kernel<8, 4, false, false> 4x1x1 352x1x1 95376',
            ],
            'bwd': [
                'bnf_bwd_reduce_wide_kernel<8, 2, false, false> 4x1x1 352x1x1 93456',
                'bnf_bwd_apply_wide_kernel<8, 2, false, false, false, false> 4x1x1 352x1x1 103696',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<4> 8x1x1 352x1x1 10640',
                'bn_apply_wide_kernel<4, 4> 8x1x1 352x1x1 45632',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<4, 4> 8x1x1 352x1x1 85248',
                'bn_bwd_apply_wide_kernel<4, 4> 8x1x1 352x1x1 108576',
            ],
        },
    },
    'skeleton_fast/2': {
        '1': {
            'fwd': [
                'bn_stats_kernel<8> 8x1x1 288x1x1 17920',
                'bnf_apply_wide_kernel<8, 2, true, false> 8x1x1 288x1x1 81936',
            ],
            'bwd': [
                'bnf_bwd_reduce_wide_kernel<8, 1, true, false> 8x1x1 288x1x1 62096',
                'bnf_bwd_apply_wide_kernel<8, 1, true, true, false, false> 8x1x1 288x1x1 72336',
            ],
            'bwd_add': [
                'bnf_bwd_reduce_wide_kernel<8, 1, true, false> 8x1x1 288x1x1 62096',
                'bnf_bwd_apply_wide_kernel<8, 1, true, true, true, false> 8x1x1 288x1x1 90256',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<8> 8x1x1 288x1x1 17920',
                'bn_apply_wide_kernel<8, 2> 8x1x1 288x1x1 74752',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<8, 1> 8x1x1 288x1x1 53888',
                'bn_bwd_apply_wide_kernel<8, 1> 8x1x1 288x1x1 64896',
            ],
            'bwd_add': [
                'bn_bwd_reduce_kernel<8, 1> 8x1x1 288x1x1 53888',
                'bn_bwd_apply_add_wide_kernel<8, 1> 8x1x1 288x1x1 82816',
            ],
        },
    },
    'skeleton_fast/3': {
        '1': {
            'fwd': [
                'bn_eval_stats_kernel 4x1x1 128x1x1 0',
                'bnf_apply_wide_kernel<8, 4, false, false> 8x1x1 288x1x1 81936',
            ],
            'bwd': [
                'bnf_bwd_reduce_wide_kernel<8, 2, false, false> 8x1x1 288x1x1 80016',
                'bnf_bwd_apply_wide_kernel<8, 2, false, false, false, false> 8x1x1 288x1x1 90256',
            ],
        },
        '0': {
            'fwd': [
                'bn_eval_stats_kernel 4x1x1 128x1x1 0',
                'bn_apply_wide_kernel<8, 4> 8x1x1 288x1x1 74752',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<8, 2> 8x1x1 288x1x1 71808',
                'bn_bwd_apply_wide_kernel<8, 2> 8x1x1 288x1x1 91776',
            ],
        },
    },
    'skeleton_fast/4': {
        '1': {
            'fwd': [
                'bn_stats_big_kernel 4x1x1 576x1x1 35840',
                'bnf_apply_wide_kernel<8, 2, true, true> 4x1x1 576x1x1 153616',
            ],
            'bwd': [
                'bnf_bwd_reduce_wide_kernel<8, 1, true, true> 4x1x1 576x1x1 115856',
                'bnf_bwd_apply_wide_kernel<8, 1, true, true, false, true> 4x1x1 576x1x1 126096',
            ],
            'bwd_add': [
                'bnf_bwd_reduce_wide_kernel<8, 1, true, true> 4x1x1 576x1x1 115856',
                'bnf_bwd_apply_wide_kernel<8, 1, true, true, true, true> 4x1x1 576x1x1 161936',
            ],
        },
        '0': REFUSED,
    },
    'skeleton_fast/5': {
        '1': {
            'fwd': [
                'bn_stats_big_kernel 4x1x1 576x1x1 35840',
                'bnf_apply_wide_kernel<8, 2, false, true> 4x1x1 576x1x1 81936',
            ],
            'bwd': [
                'bnf_bwd_reduce_wide_kernel<8, 2, false, true> 4x1x1 576x1x1 151696',
                'bnf_bwd_apply_wide_kernel<8, 2, false, false, false, true> 4x1x1 576x1x1 161936',
            ],
        },
        '0': REFUSED,
    },
    'skeleton_fast/6': {
        '1': {
            'fwd': [
                'bn_stats_kernel<4> 8x1x1 512x1x1 15400',
                'bn_apply_wide_kernel<4, 2> 8x1x1 512x1x1 64672',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<4, 2> 8x1x1 512x1x1 92528',
                'bn_bwd_apply_wide_kernel<4, 2> 8x1x1 512x1x1 109976',
            ],
            'bwd_add': [
                'bn_bwd_reduce_kernel<4, 2> 8x1x1 512x1x1 92528',
                'bn_bwd_apply_add_wide_kernel<4, 1> 8x1x1 512x1x1 71476',
            ],
        },
    },
    'skeleton_fast/7': {
        '1': {
            'fwd': [
                'bn_stats_kernel<4> 8x1x1 320x1x1 9504',
                'bnf_apply_wide_kernel<4, 4, false, false> 8x1x1 320x1x1 48272',
            ],
            'bwd': [
                'bnf_bwd_reduce_wide_kernel<4, 4, false, false> 8x1x1 320x1x1 84368',
                'bnf_bwd_apply_wide_kernel<4, 4, false, false, false, false> 8x1x1 320x1x1 94608',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<4> 8x1x1 320x1x1 9504',
                'bn_apply_wide_kernel<4, 4> 8x1x1 320x1x1 41088',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<4, 4> 8x1x1 320x1x1 76160',
                'bn_bwd_apply_wide_kernel<4, 4> 8x1x1 320x1x1 97216',
            ],
        },
    },
    'skeleton_fast/8': {
        '1': {
            'fwd': [
                'bn_stats_kernel<1> 6x1x1 480x1x1 3600',
                'bnf_apply_wide_kernel<4, 4, true, false> 3x1x1 256x1x1 67856',
            ],
            'bwd': [
                'bnf_bwd_reduce_wide_kernel<4, 4, true, false> 3x1x1 256x1x1 94736',
                'bnf_bwd_apply_wide_kernel<4, 4, true, true, false, false> 3x1x1 256x1x1 104976',
            ],
            'bwd_add': [
                'bnf_bwd_reduce_wide_kernel<4, 4, true, false> 3x1x1 256x1x1 94736',
                'bnf_bwd_apply_wide_kernel<4, 2, true, true, true, false> 3x1x1 256x1x1 76176',
            ],
        },
        '0': {
            'fwd': [
                'bn_stats_kernel<1> 6x1x1 480x1x1 3600',
                'bn_apply_wide_kernel<1, 4> 6x1x1 480x1x1 31872',
            ],
            'bwd': [
                'bn_bwd_reduce_kernel<1, 4> 6x1x1 480x1x1 43328',
                'bn_bwd_apply_wide_kernel<1, 4> 6x1x1 480x1x1 52576',
            ],
            'bwd_add': [
                'bn_bwd_reduce_kernel<1, 4> 6x1x1 480x1x1 43328',
                'bn_bwd_apply_add_wide_kernel<1, 4> 6x1x1 480x1x1 66976',
            ],
        },
    },
    'sync/parity/0': {
        '1': {
            'fwd_local': [
                'bn_stats_kernel<2> 16x1x1 416x1x1 6160',
                'bn_sync_fold_fwd_kernel 16x1x1 256x1x1 512',
            ],
            'fwd_global': [
                'bn_sync_merge_fwd_kernel 3x1x1 128x1x1 0',
                'bnf_apply_kernel<4, 4, true, false> 8x1x1 416x1x1 101136',
            ],
            'bwd_local': [
                'bnf_bwd_reduce_kernel<4, 2, true, false> 8x1x1 416x1x1 76112',
                'bn_sync_fold_bwd_kernel 16x1x1 416x1x1 640',
            ],
            'bwd_global': [
                'bnf_bwd_apply_sync_kernel<4, 2, true, true, false, false> 8x1x1 416x1x1 78544',
            ],
        },
        '0': {
            'fwd_local': [
                'bn_stats_kernel<2> 16x1x1 416x1x1 6160',
                'bn_sync_fold_fwd_kernel 16x1x1 256x1x1 512',
            ],
            'fwd_global': [
                'bn_sync_merge_fwd_kernel 3x1x1 128x1x1 0',
                'bn_apply_kernel<2, 4> 16x1x1 416x1x1 50048',
            ],
            'bwd_local': [
                'bn_bwd_reduce_kernel<2, 4> 16x1x1 416x1x1 74048',
                'bn_sync_fold_bwd_kernel 16x1x1 416x1x1 640',
            ],
            'bwd_global': [
                'bn_bwd_apply_sync_kernel<2, 4> 16x1x1 416x1x1 86752',
            ],
        },
    },
    'sync/skeleton/2': {
        '1': {
            'fwd_local': [
                'bn_stats_kernel<4> 8x1x1 352x1x1 10640',
                'bn_sync_fold_fwd_wide_kernel 8x1x1 256x1x1 2048',
            ],
            'fwd_global': [
                'bn_sync_merge_fwd_kernel 3x1x1 128x1x1 0',
                'bnf_apply_wide_kernel<8, 2, true, false> 4x1x1 352x1x1 95376',
            ],
            'bwd_local': [
                'bnf_bwd_reduce_wide_kernel<8, 1, true, false> 4x1x1 352x1x1 72176',
                'bn_sync_fold_bwd_wide_kernel 8x1x1 352x1x1 2176',
            ],
            'bwd_global': [
                'bnf_bwd_apply_sync_wide_kernel<8, 1, true, true, false, false> 4x1x1 352x1x1 82288',
            ],
        },
        '0': {
            'fwd_local': [
                'bn_stats_kernel<4> 8x1x1 352x1x1 10640',
                'bn_sync_fold_fwd_wide_kernel 8x1x1 256x1x1 2048',
            ],
            'fwd_global': [
                'bn_sync_merge_fwd_kernel 3x1x1 128x1x1 0',
                'bn_apply_wide_kernel<4, 4> 8x1x1 352x1x1 88192',
            ],
            'bwd_local': [
                'bn_bwd_reduce_kernel<4, 2> 8x1x1 352x1x1 63968',
                'bn_sync_fold_bwd_wide_kernel 8x1x1 352x1x1 2176',
            ],
            'bwd_global': [
                'bn_bwd_apply_sync_wide_kernel<4, 2> 8x1x1 352x1x1 76528',
            ],
        },
    },
}


@pytest.mark.gpu
@pytest.mark.parametrize("fast", ["1", "0"])
def test_bn_kernel_launches(fast, monkeypatch):
    monkeypatch.setenv("DSTD_BN_FAST", fast)
    for cid, case in BN_CASES.items():
        want = BN_LAUNCHES[cid].get(fast, BN_LAUNCHES[cid]['1'])
        if want == REFUSED:
            with pytest.raises(RuntimeError, match="4096 positions"):
                bn_launches(case)
        else:
            assert bn_launches(case) == want, (cid, fast)
    for cid in BN_SYNC_CASES:
        want = BN_LAUNCHES["sync/" + cid]
        assert bn_sync_launches(BN_CASES[cid]) == want.get(fast, want['1']), (cid, fast)
