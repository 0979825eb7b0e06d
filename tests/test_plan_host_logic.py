"""Host-side planning logic without a GPU: the SIMT flavour of occd_conv_plan_create needs no CUDA driver, so whole
launch plans can be BUILT (not run) on CPU tensors.  Checks the tap lists / shapes through the plan's MAC count
against the reference's published layer arithmetic (SURVEY.md section 0: 3-D UNet + CRP at config 2 = 529.9 GMAC conv
+ 4.3 GMAC bmm) and the automatic halo-exchange insertion of the X-slab partition (24 exchanges, 1/8 of the work)."""
import contextlib
import io

import pytest
import torch
import torch.nn as nn


@pytest.fixture()
def simt(monkeypatch):
    monkeypatch.setenv("OCCDEPTH_CONV_IMPL", "simt")


def _build(m, shape, slab=None):
    from occdepth_b200.engine import Plan
    plan = Plan(torch.device("cpu"), slab=slab)
    x = plan.alloc(*shape)
    with torch.no_grad():
        y = m.emit(plan, x)
    return plan, y


def test_unet3d_config2_plan_macs_and_outputs(simt):
    from occdepth_b200.models.unet3d_kitti import UNet3D
    with contextlib.redirect_stdout(io.StringIO()):
        m = UNet3D(20, nn.BatchNorm3d, (256, 256, 32), 64, 2, context_prior=True, cascade_cls=True).eval()
    plan, y = _build(m, (1, 128, 128, 16, 64))
    gmac = plan.flops / 2e9
    assert abs(gmac - (529.9 + 4.3)) / 534.2 < 0.01, gmac
    assert tuple(y["ssc_logit"].shape) == (1, 20, 256, 256, 32) and tuple(y["occ_logit"].shape) == (1, 2, 256, 256, 32)
    assert tuple(y["P_logits"].shape) == (1, 4, 512, 4096)
    assert y["x3d_l1"].dims == (1, 128, 128, 16) and y["x3d_l3"].dims == (1, 32, 32, 4)


def test_unet3d_config2_slab_plan(simt):
    from occdepth_b200.models.unet3d_kitti import UNet3D
    from occdepth_b200.parallel import SimSlabGroup
    with contextlib.redirect_stdout(io.StringIO()):
        m = UNet3D(20, nn.BatchNorm3d, (256, 256, 32), 64, 2, context_prior=True, cascade_cls=True).eval()
    full, _ = _build(m, (1, 128, 128, 16, 64))
    grp = SimSlabGroup(8, halo=3)
    plans = [_build(m, (1, 16, 128, 16, 64), slab=ctx) for ctx in (grp.ctxs[0], grp.ctxs[3])]
    for (plan, y), ctx in zip(plans, (grp.ctxs[0], grp.ctxs[3])):
        assert ctx.n_exchanges == 24 and ctx.n_gathers == 1
        assert tuple(y["ssc_logit"].shape) == (1, 20, 32, 256, 32)
        assert tuple(y["P_logits"].shape) == (1, 4, 512, 512)
        # every conv is split 8 ways; only the tiny transposed mega-context GEMM operand is replicated
        assert abs(plan.flops * 8 / full.flops - 1.0) < 0.01
    assert len(plans[0][0].ops) == len(plans[1][0].ops)
    # a slab thinner than the dilation-3 reach must be refused, not silently wrong
    grp16 = SimSlabGroup(16, halo=3)
    with pytest.raises(RuntimeError, match="slab"):
        _build(m, (1, 8, 128, 16, 64), slab=grp16.ctxs[1])


def test_unet2d_b7_plan_macs(simt):
    """2D UNet per view at 376x1370: 531.7 GMAC (encoder ~54, DecoderBN ~478), SURVEY.md section 0"""
    from occdepth_b200.models.unet2d import UNet2D
    with contextlib.redirect_stdout(io.StringIO()):
        m = UNet2D.build(out_feature=64, use_decoder=True, backbone_2d_name="tf_efficientnet_b7_ns",
                         return_up_feats=1).eval()
    plan, y = _build(m, (1, 1, 376, 1370, 3))
    dw = 2.7       # depthwise MACs are not tensor-core launches (not in plan.flops)
    gmac = plan.flops / 2e9
    assert abs(gmac + dw - 531.7) / 531.7 < 0.02, gmac
    assert y["1_1"].dims == (1, 1, 376, 1370) and y["1_8"].dims == (1, 1, 47, 172) and y["1_16"].dims == (1, 1, 24, 86)


def test_occdepth_config2_plan(simt, monkeypatch):
    """the whole forward plan at the benchmark configuration: ~3.2 TFLOP of tensor-core launches (SURVEY.md section 0:
    2 x 531.7 GMAC 2D + 529.9 + 4.3 GMAC 3D), one fused lift launch, logits in the reference's NCDHW layout"""
    import bench
    monkeypatch.setenv("OCCDEPTH_CUDA_GRAPH", "0")
    m = bench.build_model()
    N = 128 * 128 * 16
    plan, img, pix, fov, out, depth0, n_lo, view_sel = m._build(1, 2, bench.IMG_H, bench.IMG_W, N, 1,
                                                                 torch.device("cpu"), {})
    assert view_sel is None
    gmac = plan.flops / 2e9
    assert abs(gmac + 2 * 2.7 - (2 * 531.7 + 529.9 + 4.3)) / 1597.6 < 0.02, gmac
    assert sum(1 for op in plan.ops if getattr(op, "name", "") == "sfa_lift") == 1
    assert tuple(out["ssc_logit"].shape) == (1, 20, 256, 256, 32)
    assert img.dims == (2, 1, bench.IMG_H, bench.IMG_W) and tuple(pix.shape) == (1, 2, N, 1, 2)
    assert len(plan.ops) < 500      # both views batched, SE + projection batched over images


def test_occdepth_config2_slab_plan_shards_2d_net_by_view(simt, monkeypatch):
    """X-slab partition of one frame over 8 ranks (BASELINE configs[2]): the 2D net runs ONE view per rank (ranks 0-3
    view 0, ranks 4-7 view 1) and one all-gather hands every rank both views' feature maps; the lift and the 3D net
    work on this rank's 16 of 128 X-planes."""
    import bench
    from occdepth_b200.parallel import SimSlabGroup
    monkeypatch.setenv("OCCDEPTH_CUDA_GRAPH", "0")
    m = bench.build_model()
    N = 128 * 128 * 16
    full = m._build(1, 2, bench.IMG_H, bench.IMG_W, N, 1, torch.device("cpu"), {})[0]
    grp = SimSlabGroup(8, halo=3)
    ents = {}
    for r in (1, 6):
        m.__dict__["slab_ctx"] = grp.ctxs[r]
        ents[r] = m._build(1, 2, bench.IMG_H, bench.IMG_W, N, 1, torch.device("cpu"), {})
    m.__dict__.pop("slab_ctx")
    assert ents[1][7] == 0 and ents[6][7] == 1                      # which view each rank's 2D net processes
    for r, (plan, img, pix, fov, out, depth0, n_lo, view_sel) in ents.items():
        assert img.dims == (1, 1, bench.IMG_H, bench.IMG_W)          # one view
        assert tuple(pix.shape) == (1, 2, N // 8, 1, 2) and n_lo == r * (N // 8)
        names = [getattr(op, "name", "") for op in plan.ops]
        assert names.count("all_gather") == 2                       # 2D feature maps + CRP mega-context
        assert names.index("all_gather") < names.index("sfa_lift")
        # per-rank tensor-core work: half of the 2D net (one of two views) + an eighth of the 3D net
        want = (531.7 - 2.7) + (529.9 + 4.3) / 8
        assert abs(plan.flops / 2e9 - want) / want < 0.03, plan.flops / 2e9
        assert tuple(out["ssc_logit"].shape) == (1, 20, 32, 256, 32)
    assert len(ents[1][0].ops) == len(ents[6][0].ops)
    assert full.flops > 2.5 * ents[1][0].flops


def test_variant_eligibility_rules():
    """host-side kernel selection rules (engine.py) on the shapes they were written for"""
    from occdepth_b200 import engine as E
    t333 = [(0, a, b, c) for a in (-1, 0, 1) for b in (-1, 0, 1) for c in (-1, 0, 1)]
    t333_d2 = [(0, 2 * a, 2 * b, 2 * c) for a in (-1, 0, 1) for b in (-1, 0, 1) for c in (-1, 0, 1)]
    two_src = [(s, 0, b, c) for s in (0, 1) for b in (-1, 0, 1) for c in (-1, 0, 1)]
    assert E.tcx_eligible(t333, (1, 1, 1), 80) and E.tcx_eligible(two_src, (1, 1, 1), 80)
    assert not E.tcx_eligible(t333_d2, (1, 1, 1), 64)        # W dilation 2: per-tap kernel has no sub-grids
    assert not E.tcx_eligible(t333, (1, 1, 2), 64) and not E.tcx_eligible(t333, (1, 1, 1), 96)
    assert not E.tcx_eligible(t333, (1, 1, 1), 32)           # narrow outputs: the halo kernel's shapes
    # K chunk = one swizzled smem row of 32 / 64 / 128 bytes
    assert [E.chunk_channels(c, 2) for c in (3, 16, 17, 32, 33, 64, 65, 2784)] == [16, 16, 32, 32, 64, 64, 64, 64]
    assert [E.chunk_channels(c, 4) for c in (3, 8, 9, 16, 17, 32, 33, 2784)] == [8, 8, 16, 16, 32, 32, 32, 32]
    # TF32 rounding: ties away from zero on the 13 dropped mantissa bits == cvt.rna.tf32.f32
    t = torch.tensor([1.0, 1.0 + 2.0 ** -11, 1.0 + 2.0 ** -11 + 2.0 ** -20, -(1.0 + 2.0 ** -11), 3.0e-39, 65504.0])
    r = E.round_tf32_(t.clone())
    assert r.tolist()[:4] == [1.0, 1.0 + 2.0 ** -10, 1.0 + 2.0 ** -10, -(1.0 + 2.0 ** -10)]
    assert torch.equal(r.view(torch.int32) & 0x1FFF, torch.zeros(6, dtype=torch.int32))


# the tensor-map encode is the first step of plan creation that needs a driver: without one its entry point is
# missing; with one it is called and refuses the host tensors these tests pass (no CUDA context is current)
ENCODE_ERROR = ("cuTensorMapEncodeTiled\\(source \\d+\\) failed" if torch.cuda.is_available()
                else "cuTensorMapEncodeTiled unavailable")


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
def test_auto_impl_selection_reaches_tensor_map_encode(monkeypatch, precision):
    """'auto' mode (the GPU default) on the CPU: selection rules + plan geometry run; the first thing that needs a
    driver is cuTensorMapEncodeTiled, and the product must say so instead of falling back to anything"""
    from occdepth_b200.engine import CL, Plan
    monkeypatch.delenv("OCCDEPTH_CONV_IMPL", raising=False)
    shapes = [((4, 8, 40), 32, 32, (3, 3, 3)), ((1, 40, 90), 160, 160, (1, 3, 3)), ((1, 20, 30), 48, 288, (1, 1, 1)),
              ((1, 188, 685), 80, 80, (1, 3, 3))]
    for dims, ci, co, k in shapes:
        plan = Plan(torch.device("cpu"), precision=precision)
        x = plan.alloc(2, dims[0], dims[1], dims[2], ci)
        with pytest.raises(RuntimeError, match=ENCODE_ERROR):
            plan.conv(x, torch.randn(co, ci, *k), torch.randn(co), padding=tuple(kk // 2 for kk in k))


def test_tap_group_plans_are_validated_on_the_host(monkeypatch):
    """tap groups (the transposed conv's eight phases as ONE launch): the grouped plan passes the host-side geometry
    and reaches the tensor-map encode (the first step that needs a driver); malformed group tables, a second output or
    a non-TC kernel are refused by occd_conv_plan_create with a message"""
    import ctypes as C
    from occdepth_b200 import _lib
    from occdepth_b200.engine import ConvOp, Plan
    monkeypatch.delenv("OCCDEPTH_CONV_IMPL", raising=False)
    plan = Plan(torch.device("cpu"), precision="tf32")
    x = plan.alloc(1, 4, 6, 8, 32)
    with pytest.raises(RuntimeError, match=ENCODE_ERROR):
        plan.conv_transpose_k3s2(x, torch.randn(32, 16, 3, 3, 3), torch.randn(16), act="relu")
    out = plan.alloc(1, 8, 12, 16, 16)
    taps = [(0, 0, 0, 0), (0, 0, 0, 1), (0, 0, 1, 0)]
    ws = [torch.randn(16, 32) for _ in taps]
    L = _lib.lib()

    def create(groups, **kw):
        with pytest.raises(RuntimeError) as ei:
            ConvOp([x], taps, ws, torch.randn(16), (4, 6, 8), out0=out, omul=(2, 2, 2), full_dims=(8, 12, 16),
                   groups=groups, **kw)
        return str(ei.value)

    assert "cuTensorMapEncodeTiled" in create([(2, (1, 1, 1)), (1, (0, 0, 0))])          # well-formed
    assert "tap groups" in create([(2, (2, 0, 0)), (1, (0, 0, 0))])                         # oadd >= omul
    assert "tap groups" in create([(2, (1, 1, 1)), (1, (0, 0, 0))], out1=plan.alloc(1, 8, 12, 16, 16), out1_mode="cl")
    d = _lib.ConvDesc()
    d.impl, d.n_groups = _lib.CONV_IMPL_SIMT, 2
    h = C.c_void_p()
    assert L.occd_conv_plan_create(C.byref(d), C.byref(h)) != 0


def test_widened_rows_fail_loudly_without_cuda():
    """no CPU fallback anywhere: the data-pipeline and post-processing entry points refuse to run without a GPU"""
    import numpy as np
    from occdepth_b200 import data
    from occdepth_b200.models.OccDepth import OccDepth
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    with pytest.raises(RuntimeError, match="CUDA"):
        data.vox2pix(np.eye(4), np.eye(3), np.zeros(3), 0.4, 64, 48, (3.2, 3.2, 1.6), 0)
    with pytest.raises(RuntimeError, match="CUDA"):
        data.normalize_rgb(np.zeros((4, 4, 3), dtype=np.uint8), 4, 4)
    with pytest.raises(RuntimeError, match="CUDA"):
        OccDepth.class_map(torch.zeros(1, 20, 2, 2, 2))
    # host-side helpers shared with the tests are plain numpy
    assert tuple(data.volume_dims(np.array([0, -25.6, -2.0]), 0.4, (51.2, 51.2, 6.4))) == (128, 128, 16)
    assert [len(p) for p in data.PIXEL_PATTERNS] == [1, 5, 5, 9, 9, 13, 25, 8, 21]
