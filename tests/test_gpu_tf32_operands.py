"""The tf32 storage contract of the convolution operands.

`OCCD_DTYPE_F32` buffers are fp32 storage holding TF32 values (include/occdepth_b200.h): every producer rounds at the
store, and the `tcgen05 kind::tf32` convolutions read them as MMA operands.  These tests build small tf32 models, run
one forward, then replay the cached plan's launches one at a time.  Before every convolution they check that each
source window (the whole buffer's [coff, coff + C), halo planes included) and the weights (CRP weights are produced at
run time) are finite and equal to their TF32 rounding, so a producer that stores unrounded fp32 is named at the first
convolution that reads it.  After the walk the outputs must equal the forward's bit for bit, which also checks that
nothing carries over from one replay to the next.  In bf16 the same walk checks finiteness.
"""
import copy

import pytest
import torch
import torch.nn as nn

from oracle import ref_import, synth

import gpu_cases as G

pytestmark = pytest.mark.gpu


def _occdepth_kitti_flosp():
    from occdepth_b200.models.OccDepth import OccDepth
    full, ps = (32, 32, 16), 2
    cfg = synth.occdepth_cfg(dataset="kitti", full_scene_size=full, project_scale=ps, feature=32, feature_2d_oc=32,
                             n_classes=20, cascade_cls=True, backbone_2d_name="tf_efficientnet_b3_ns")
    with ref_import.quiet():
        m = OccDepth(["c"] * 20, torch.ones(20), full_scene_size=full, project_res=["1", "2", "4", "8"],
                     config=cfg).eval()
    synth.randomize_bn_(m)
    H, W = 33, 49
    img = torch.randn(1, 2, 3, H, W, generator=torch.Generator().manual_seed(0))
    N = (full[0] // ps) * (full[1] // ps) * (full[2] // ps)
    pix, fov = synth.random_indices(N, W, H, n_views=2, P=1, seed=5, margin=(10, 6))
    return m, {"img": img, "projected_pix_%d" % ps: [pix], "fov_mask_%d" % ps: [fov]}


def _occdepth_flosp_depth():
    from occdepth_b200.models.OccDepth import OccDepth
    import occdepth_b200.models.flosp_depth.flosp_depth as fd
    full, ps = (32, 32, 16), 2
    H, W = 40, 96
    saved = copy.deepcopy(fd.flosp_depth_conf_map["kitti"])
    try:
        fd.flosp_depth_conf_map["kitti"].update(final_dim=(H, W), x_bound=[0, 6.4, 0.2], y_bound=[-3.2, 3.2, 0.2],
                                                z_bound=[-2, 1.2, 0.2], d_bound=[1.0, 9.0, 0.5])
        cfg = synth.occdepth_cfg(full_scene_size=full, project_scale=ps, feature=32, feature_2d_oc=32, n_classes=8,
                                 backbone_2d_name="tf_efficientnet_b3_ns", trans_2d_to_3d="flosp_depth",
                                 use_stereo_depth_gt=True)
        with ref_import.quiet():
            m = OccDepth(["c"] * 8, torch.ones(8), full_scene_size=full, project_res=["1", "2", "4", "8"],
                         config=cfg).eval()
    finally:
        fd.flosp_depth_conf_map["kitti"].clear()
        fd.flosp_depth_conf_map["kitti"].update(saved)
    synth.seed_weights_(m, 9)
    K, Ts = synth.kitti_calib(W, H, focal=60.0)
    img = torch.randn(1, 2, 3, H, W, generator=torch.Generator().manual_seed(1))
    pix, fov = synth.random_indices(16 * 16 * 8, W, H, n_views=2, P=1, seed=5, margin=(10, 6))
    return m, {"img": img, "projected_pix_2": [pix], "fov_mask_2": [fov],
               "cam_k": [torch.from_numpy(K).unsqueeze(0).repeat(2, 1, 1)],
               "T_velo_2_cam": [torch.stack([torch.from_numpy(t) for t in Ts])],
               "ida_mats": [torch.eye(4).unsqueeze(0).repeat(2, 1, 1)]}


def _occdepth_nyu_virtual():
    from occdepth_b200.models.OccDepth import OccDepth
    from oracle.reference_cases import nyu_virtual_batch
    full = (12, 8, 12)
    cfg = synth.occdepth_cfg(dataset="NYU", full_scene_size=full, project_scale=1, feature=16, feature_2d_oc=16,
                             n_classes=6, cascade_cls=False, backbone_2d_name="tf_efficientnet_b3_ns")
    with ref_import.quiet():
        m = OccDepth(["c"] * 6, torch.ones(6), full_scene_size=full, project_res=["1", "2", "4", "8"],
                     config=cfg).eval()
    synth.seed_weights_(m, 3)
    return m, nyu_virtual_batch(32, 64, full)


def _unet3d():
    from occdepth_b200.models.unet3d_kitti import UNet3D
    full, ps, f = (32, 32, 16), 2, 32
    m = UNet3D(20, nn.BatchNorm3d, full, f, ps, context_prior=True, cascade_cls=True, occluded_cls=True).eval()
    synth.randomize_bn_(m)
    return m, {"x3d": torch.randn(1, f, 16, 16, 8, generator=torch.Generator().manual_seed(2))}


MODELS = {"kitti_flosp": _occdepth_kitti_flosp, "flosp_depth": _occdepth_flosp_depth,
          "nyu_virtual": _occdepth_nyu_virtual, "unet3d": _unet3d}


def _cuda_batch(batch):
    return {k: (v.cuda() if k in ("img", "x3d") else v) for k, v in batch.items()}


def _plan_outputs(m):
    """(plan, function returning the outputs the cached plan's buffers hold now)"""
    from occdepth_b200.models._base import _to_planar
    from occdepth_b200.models.OccDepth import OccDepth
    (ent,) = m._plans().values()
    if isinstance(m, OccDepth):
        plan, out = ent[0], ent[4]

        def outputs():
            res = _to_planar(out, False)
            if m.with_depth_gt and m.trans_2d_to_3d == "flosp_depth":
                res["depth_pred"] = m.flosp_depth.depth_prob()
            return res
        return plan, outputs
    plan, _, y = ent
    return plan, lambda: _to_planar(y, False)


def _bad(t, precision):
    """None if t satisfies the storage contract, else what is wrong"""
    if not bool(torch.isfinite(t).all()):
        return "not finite"
    if precision == "tf32":
        t = t.contiguous()
        n = int((t != G.tf32r(t)).sum())
        if n:
            return "%d of %d values are not TF32" % (n, t.numel())
    return None


@pytest.mark.parametrize("precision", G.PRECISIONS)
@pytest.mark.parametrize("model", list(MODELS))
def test_conv_operands_keep_the_storage_contract(model, precision):
    from occdepth_b200 import _lib
    from occdepth_b200.engine import ConvOp
    torch.manual_seed(0)
    m, batch = MODELS[model]()
    m = m.cuda().set_precision(precision)
    with torch.no_grad():
        got = m(_cuda_batch(batch))
    plan, outputs = _plan_outputs(m)
    st = _lib.stream_ptr()
    n_conv = 0
    for op in plan.ops:
        if isinstance(op, ConvOp):
            torch.cuda.synchronize()
            n_conv += 1
            for si, s in enumerate(op._keep[0]):
                why = _bad(s.buf[..., s.coff:s.coff + s.C], precision)
                assert why is None, "conv %r: source %d: %s" % (op.name, si, why)
            why = _bad(op.weight, precision)
            assert why is None, "conv %r: weights: %s" % (op.name, why)
        op.run(st)
    torch.cuda.synchronize()
    assert n_conv > 10
    after = outputs()
    assert set(after) == set(got)
    for k in got:
        assert torch.equal(after[k], got[k]), "%s differs after the op-by-op replay" % k
