"""Kernel-path and workspace decisions of the DSTD-GC entry points.

Without a GPU: whether a call keeps ``xa``, and the workspace sizes of every entry point, for the unit shapes of the
parity tests and a (P, K) sweep across the 40-wide specialised tiles, under the default switches and each documented
switch setting (set in-process: the library reads them per call).  The sizes and the xa decision do not depend on the
switches, so a caller that sized its buffers before flipping one still hands over enough workspace.

On the GPU: the kernels one forward + backward launches, per shape and switch setting.

TABLE and KERNELS hold what the library did before these decisions were moved into one plan (api.cu gc_plan); a change
to either is a change of what the library computes, allocates or launches."""
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
