"""2D UNet (EfficientNet encoder + DecoderBN) and the whole OccDepth.forward on CUDA vs the CPU fp32 oracle."""
import pytest
import torch

from oracle import functional as OF
from oracle import ref_import, synth

import gpu_cases as G

pytestmark = pytest.mark.gpu
PREC = pytest.mark.parametrize("precision", G.PRECISIONS)

# stated tolerances relative to max-abs of the CPU fp32 oracle tensor, per precision mode (<= 2x the values measured on
# B200, profiles/r02_parity_measured.jsonl): "tf32" = TF32 operands / fp32 accumulate / TF32-valued fp32 activations
# (the reference-precision mode), "bf16" = bf16 operands and activations
# measured: 2D net tf32 <= 6.9e-4 / bf16 <= 6.4e-3; small full forwards tf32 <= 1.3e-3 / bf16 <= 8.5e-3, arg-max
# agreement tf32 >= 0.99958, bf16 >= 0.9985
TOL_2D = {"tf32": 1.4e-3, "bf16": 1.3e-2}
TOL_E2E = {"tf32": 2.5e-3, "bf16": 1.7e-2}
TOL_ARGMAX = {"tf32": 0.999, "bf16": 0.997}


def _rel(g, w):
    return float((g.float().cpu() - w).abs().max() / w.abs().max().clamp_min(1e-6))


@PREC
@pytest.mark.parametrize("backbone,hw", [("tf_efficientnet_b3_ns", (38, 45)), ("tf_efficientnet_b7_ns", (33, 49))])
def test_unet2d(backbone, hw, precision):
    from occdepth_b200.models.unet2d import UNet2D
    torch.manual_seed(0)
    with ref_import.quiet():
        m = UNet2D.build(out_feature=32, use_decoder=True, backbone_2d_name=backbone, return_up_feats=1).eval()
    synth.randomize_bn_(m)
    sd = {"net_rgb." + k: v.clone() for k, v in m.state_dict().items()}
    x = torch.randn(1, 3, *hw)
    with torch.no_grad():
        want = OF.unet2d(sd, "net_rgb", x, backbone, 1)
        got = m.cuda().set_precision(precision)(x.cuda())
    assert set(got.keys()) == set(want.keys())
    G.record("unet2d[%s]" % backbone, precision, **{k: _rel(got[k], want[k]) for k in want})
    for k in want:
        assert got[k].shape == want[k].shape, k
        assert _rel(got[k], want[k]) <= TOL_2D[precision], (k, _rel(got[k], want[k]))


@PREC
@pytest.mark.parametrize("dataset", ["kitti", "NYU"])
def test_occdepth_forward_small(dataset, precision):
    """config-1-like plumbing case: tiny stereo pair, both decoders, CRP on; max-abs-diff of the voxel logits."""
    from occdepth_b200.models.OccDepth import OccDepth
    torch.manual_seed(0)
    if dataset == "kitti":
        full, ps, ncls, casc = (32, 32, 16), 2, 20, True
    else:
        full, ps, ncls, casc = (20, 12, 20), 1, 12, False
    cfg = synth.occdepth_cfg(dataset=dataset, full_scene_size=full, project_scale=ps, feature=32, feature_2d_oc=32,
                             n_classes=ncls, cascade_cls=casc, backbone_2d_name="tf_efficientnet_b3_ns")
    with ref_import.quiet():
        m = OccDepth(["c"] * ncls, torch.ones(ncls), full_scene_size=full, project_res=["1", "2", "4", "8"],
                     config=cfg).eval()
    synth.randomize_bn_(m)
    H, W = 33, 49
    g = torch.Generator().manual_seed(0)
    img = torch.randn(1, 2, 3, H, W, generator=g)
    N = (full[0] // ps) * (full[1] // ps) * (full[2] // ps)
    pix, fov = synth.random_indices(N, W, H, n_views=2, P=1, seed=5, margin=(10, 6))
    batch = {"img": img, "projected_pix_%d" % ps: [pix], "fov_mask_%d" % ps: [fov]}
    ocfg = dict(cfg)
    ocfg["project_res"] = ["1", "2", "4", "8"]
    with torch.no_grad():
        want = OF.occdepth_forward({k: v.clone() for k, v in m.state_dict().items()}, batch, ocfg)
        got = m.cuda().set_precision(precision)({"img": img.cuda(), "projected_pix_%d" % ps: [pix],
                                                 "fov_mask_%d" % ps: [fov]})
    assert set(got.keys()) == set(want.keys())
    agree = float((got["ssc_logit"].argmax(1).cpu() == want["ssc_logit"].argmax(1)).float().mean())
    G.record("occdepth_forward_small[%s]" % dataset, precision, argmax=agree,
             **{k: _rel(got[k], want[k]) for k in want})
    for k in want:
        assert got[k].shape == want[k].shape, k
        assert _rel(got[k], want[k]) <= TOL_E2E[precision], (k, _rel(got[k], want[k]))
    assert agree >= TOL_ARGMAX[precision], agree


def _flosp_conf(H, W):
    import copy
    from occdepth_b200.models.flosp_depth import flosp_depth_conf_map
    conf = copy.deepcopy(flosp_depth_conf_map["kitti"])
    conf.update(scene_size=(64, 64, 8), project_scale=2, return_depth=True, final_dim=(H, W), output_channels=16,
                x_bound=[0, 12.8, 0.2], y_bound=[-6.4, 6.4, 0.2], z_bound=[-2, -0.4, 0.2], d_bound=[2.0, 18.0, 0.5],
                depth_net_conf=dict(in_channels=16, mid_channels=32))
    return conf


@PREC
def test_flosp_depth_module(precision):
    """FlospDepth drop-in (DepthNet on tcgen05 + fused frustum sampling kernel) vs the CPU oracle"""
    from occdepth_b200.models.flosp_depth import FlospDepth
    torch.manual_seed(0)
    H, W = 96, 320
    conf = _flosp_conf(H, W)
    m = synth.seed_weights_(FlospDepth(**conf), 5).eval()
    K, Ts = synth.kitti_calib(W, H, focal=220.0)
    cam_k = [torch.from_numpy(K).unsqueeze(0).repeat(2, 1, 1)]
    T = [torch.stack([torch.from_numpy(t) for t in Ts])]
    ida = [torch.eye(4).unsqueeze(0).repeat(2, 1, 1)]
    feat = torch.randn(1, 2, 16, H // 8, W // 8)
    with torch.no_grad():
        want, want_d = OF.flosp_depth({"f." + k: v.clone() for k, v in m.state_dict().items()}, "f", feat, cam_k, T, ida,
                                      conf)
        got, got_d = m.cuda().set_precision(precision)(feat.cuda(), cam_k, T, ida, None)
    assert float((want > 0).float().mean()) > 0.2
    G.record("flosp_depth_module", precision, depth=_rel(got_d, want_d), prior=_rel(got, want))
    assert _rel(got_d, want_d) <= TOL_E2E[precision], _rel(got_d, want_d)
    assert _rel(got, want) <= TOL_E2E[precision], _rel(got, want)


@PREC
def test_occdepth_forward_flosp_depth(precision):
    """OccDepth.forward with trans_2d_to_3d="flosp_depth" (the README-default configs): lift x depth prior x 100"""
    from occdepth_b200.models.OccDepth import OccDepth
    import occdepth_b200.models.flosp_depth.flosp_depth as fd
    import copy
    torch.manual_seed(0)
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
        conf = copy.deepcopy(m.flosp_depth_conf)
    finally:
        fd.flosp_depth_conf_map["kitti"].clear()
        fd.flosp_depth_conf_map["kitti"].update(saved)
    synth.seed_weights_(m, 9)
    K, Ts = synth.kitti_calib(W, H, focal=60.0)
    img = torch.randn(1, 2, 3, H, W)
    N = 16 * 16 * 8
    pix, fov = synth.random_indices(N, W, H, n_views=2, P=1, seed=5, margin=(10, 6))
    batch = {"img": img, "projected_pix_2": [pix], "fov_mask_2": [fov],
             "cam_k": [torch.from_numpy(K).unsqueeze(0).repeat(2, 1, 1)],
             "T_velo_2_cam": [torch.stack([torch.from_numpy(t) for t in Ts])],
             "ida_mats": [torch.eye(4).unsqueeze(0).repeat(2, 1, 1)]}
    ocfg = dict(cfg)
    ocfg.update(project_res=["1", "2", "4", "8"], flosp_depth_conf=conf, with_depth_gt=True)
    with torch.no_grad():
        want = OF.occdepth_forward({k: v.clone() for k, v in m.state_dict().items()}, batch, ocfg)
        b2 = dict(batch)
        b2["img"] = img.cuda()
        got = m.cuda().set_precision(precision)(b2)
    assert set(got.keys()) == set(want.keys())
    G.record("occdepth_forward_flosp_depth", precision,
             **{k: _rel(got[k], want[k]) for k in ("ssc_logit", "occ_logit", "depth_pred")})
    for k in ("ssc_logit", "occ_logit", "depth_pred"):
        assert _rel(got[k], want[k]) <= TOL_E2E[precision], (k, _rel(got[k], want[k]))


@PREC
def test_occdepth_forward_nyu_virtual_view(precision):
    """config-4-type path: single RGB view + gt_depth -> virtual right view kernel -> lift -> NYU 3D net"""
    from occdepth_b200.models.OccDepth import OccDepth
    from oracle.reference_cases import nyu_virtual_batch
    torch.manual_seed(0)
    full = (12, 8, 12)
    cfg = synth.occdepth_cfg(dataset="NYU", full_scene_size=full, project_scale=1, feature=16, feature_2d_oc=16,
                             n_classes=6, cascade_cls=False, backbone_2d_name="tf_efficientnet_b3_ns")
    with ref_import.quiet():
        m = OccDepth(["c"] * 6, torch.ones(6), full_scene_size=full, project_res=["1", "2", "4", "8"],
                     config=cfg).eval()
    synth.seed_weights_(m, 3)
    batch = nyu_virtual_batch(32, 64, full)
    ocfg = dict(cfg)
    ocfg["project_res"] = ["1", "2", "4", "8"]
    with torch.no_grad():
        want = OF.occdepth_forward({k: v.clone() for k, v in m.state_dict().items()}, batch, ocfg)
        b2 = dict(batch)
        b2["img"] = batch["img"].cuda()
        got = m.cuda().set_precision(precision)(b2)
    assert set(got.keys()) == set(want.keys())
    G.record("occdepth_forward_nyu_virtual_view", precision, **{k: _rel(got[k], want[k]) for k in want})
    for k in want:
        assert _rel(got[k], want[k]) <= TOL_E2E[precision], (k, _rel(got[k], want[k]))


@PREC
def test_occdepth_infer_mode_flosp_depth(precision):
    """SURVEY 8f row 3, the reference's deployment route: OccDepth(infer_mode=True) disables the CRP and the
    training-only outputs (OccDepth.py:82-84, unet3d_kitti.py:108-125) and FlospDepth consumes caller-supplied sampling
    grids + scaled pixel sizes instead of camera matrices (OccDepth.py:310-317, flosp_depth.py:564-565).  The grids fed
    here are what the reference's FrustumGridGenerator produces for the same cameras (oracle.frustum_grid), so the
    result must equal the oracle's infer_mode forward."""
    from occdepth_b200.models.OccDepth import OccDepth
    import occdepth_b200.models.flosp_depth.flosp_depth as fd
    import copy
    torch.manual_seed(0)
    full, ps = (32, 32, 16), 2
    H, W = 40, 96
    saved = copy.deepcopy(fd.flosp_depth_conf_map["kitti"])
    try:
        fd.flosp_depth_conf_map["kitti"].update(final_dim=(H, W), x_bound=[0, 6.4, 0.2], y_bound=[-3.2, 3.2, 0.2],
                                                z_bound=[-2, 1.2, 0.2], d_bound=[1.0, 9.0, 0.5])
        cfg = synth.occdepth_cfg(full_scene_size=full, project_scale=ps, feature=32, feature_2d_oc=32, n_classes=8,
                                 backbone_2d_name="tf_efficientnet_b3_ns", trans_2d_to_3d="flosp_depth")
        with ref_import.quiet():
            m = OccDepth(["c"] * 8, torch.ones(8), full_scene_size=full, project_res=["1", "2", "4", "8"],
                         config=cfg, infer_mode=True).eval()
        conf = copy.deepcopy(m.flosp_depth_conf)
    finally:
        fd.flosp_depth_conf_map["kitti"].clear()
        fd.flosp_depth_conf_map["kitti"].update(saved)
    synth.seed_weights_(m, 9)
    K, Ts = synth.kitti_calib(W, H, focal=60.0)
    img = torch.randn(1, 2, 3, H, W)
    N = 16 * 16 * 8
    pix, fov = synth.random_indices(N, W, H, n_views=2, P=1, seed=5, margin=(10, 6))
    cam_k = [torch.from_numpy(K).unsqueeze(0).repeat(2, 1, 1)]
    T = [torch.stack([torch.from_numpy(t) for t in Ts])]
    ida = [torch.eye(4).unsqueeze(0).repeat(2, 1, 1)]
    batch = {"img": img, "projected_pix_2": [pix], "fov_mask_2": [fov], "cam_k": cam_k, "T_velo_2_cam": T,
             "ida_mats": ida}
    ocfg = dict(cfg)
    ocfg.update(project_res=["1", "2", "4", "8"], flosp_depth_conf=conf, infer_mode=True)
    # what a deployment precomputes on the host: per-camera sampling grids and the scaled pixel size
    bounds = [conf["x_bound"], conf["y_bound"], conf["z_bound"]]
    pc_min = torch.tensor([b[0] for b in bounds], dtype=torch.float32)
    pc_max = torch.tensor([b[1] for b in bounds], dtype=torch.float32)
    gs = [int((b[1] - b[0]) / b[2] / ps) for b in bounds]
    nb = int((conf["d_bound"][1] - conf["d_bound"][0]) / conf["d_bound"][2])
    grids, sps = [], []
    for v in range(2):
        K4 = torch.zeros(1, 4, 4)
        K4[0, :3, :3] = cam_k[0][v].float()
        K4[0, 3, 3] = 1
        grids.append(OF.frustum_grid(gs, pc_min, pc_max, T[0][v].float(), K4[0], ida[0][v], (H, W), nb,
                                     conf["d_bound"][0], conf["d_bound"][1]))
        inv = torch.inverse(K4[0])
        sps.append(torch.norm(torch.stack([inv[0, 0], inv[1, 1]])) * 1000.0)
    with torch.no_grad():
        want = OF.occdepth_forward({k: v.clone() for k, v in m.state_dict().items()}, batch, ocfg)
        b2 = {"img": img.cuda(), "projected_pix_2": [pix], "fov_mask_2": [fov], "grids": [g.cuda() for g in grids],
              "scaled_pixel_size": torch.stack(sps).reshape(2, 1).cuda()}
        got = m.cuda().set_precision(precision)(b2)
    assert set(got.keys()) == set(want.keys()) == {"ssc_logit"}
    G.record("occdepth_infer_mode_flosp_depth", precision, ssc_logit=_rel(got["ssc_logit"], want["ssc_logit"]))
    assert _rel(got["ssc_logit"], want["ssc_logit"]) <= TOL_E2E[precision]
