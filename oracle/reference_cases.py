"""Seeded cases that pin oracle/functional.py against the UNMODIFIED reference (tests/test_oracle_vs_reference.py).

Each builder takes a namespace of model modules: the reference's (`reference_modules()`, run by oracle/gen_golden.py
to record tests/golden/reference_outputs.pt) or this package's (`product_modules()`).  Under the same seed both
construct the same state_dict, so in the test this package's modules serve only as parameter containers; the
recorded `state_sum` of every case checks that they still do.
"""
import contextlib
import copy
import io
import types

import torch
import torch.nn as nn

from . import synth

SFA_CASES = [("kitti", 2, 1), ("kitti", 1, 1), ("NYU", 2, 1), ("kitti", 2, 5), ("kitti", 3, 1)]
VOX2PIX_PATTERNS = [0, 1, 3, 6, 8]
PROJECT_RES = ["1", "2", "4", "8"]


def product_modules():
    from occdepth_b200.models import OccDepth, SFA, modules, unet2d, unet3d_kitti, unet3d_nyu
    from occdepth_b200.models.flosp_depth import FlospDepth, flosp_depth_conf_map
    return types.SimpleNamespace(SFA=SFA, modules=modules, unet3d_kitti=unet3d_kitti, unet3d_nyu=unet3d_nyu,
                                 unet2d=unet2d, OccDepth=OccDepth, FlospDepth=FlospDepth,
                                 flosp_depth_conf_map=flosp_depth_conf_map)


def reference_modules():
    from . import ref_import
    r = ref_import.modules()
    import occdepth.models.flosp_depth as rfd
    return types.SimpleNamespace(SFA=r.SFA, modules=r.modules, unet3d_kitti=r.unet3d_kitti, unet3d_nyu=r.unet3d_nyu,
                                 unet2d=r.unet2d, OccDepth=r.OccDepth, FlospDepth=r.flosp_depth.FlospDepth,
                                 flosp_depth_conf_map=rfd.flosp_depth_conf_map)


def state_sum(*modules):
    """float64 sum and absolute sum of every floating-point state_dict entry"""
    s = a = 0.0
    for m in modules:
        for t in m.state_dict().values():
            if t.dtype.is_floating_point:
                s += float(t.double().sum())
                a += float(t.double().abs().sum())
    return s, a


def sample_index(n, k=512):
    """k distinct flat indices spread over a tensor of n > k elements: a fixed stride modulo n (1000003 is prime,
    so the indices are distinct unless n is a multiple of it)"""
    assert n > k and n % 1000003 != 0
    return torch.arange(k, dtype=torch.int64) * 1000003 % n


def _quiet():
    return contextlib.redirect_stdout(io.StringIO())


def sfa(dataset, V, P):
    torch.manual_seed(0)
    scene, ps = (16, 12, 8), 2
    S = [s // ps for s in scene]
    N = S[0] * S[1] * S[2]
    C, h, w = 16, 11, 23
    x2d = torch.randn(V, C, h, w)
    pix, fov = synth.random_indices(N, w, h, n_views=V, P=P, seed=3, margin=(5, 4))
    return dict(x2d=x2d, pix=pix, fov=fov, scene=scene, dataset=dataset, ps=ps)


def bottleneck(ns):
    """Process / Downsample / Upsample blocks and their input"""
    torch.manual_seed(0)
    with _quiet():
        proc = ns.modules.Process(16, nn.BatchNorm3d, 0.1, dilations=[1, 2, 3]).eval()
        down = ns.modules.Downsample(16, nn.BatchNorm3d, 0.1).eval()
        up = ns.modules.Upsample(32, 16, nn.BatchNorm3d, 0.1).eval()
    for m in (proc, down, up):
        synth.randomize_bn_(m)
    return proc, down, up, torch.randn(1, 16, 8, 10, 6)


def unet3d(ns, which):
    torch.manual_seed(0)
    with _quiet():
        if which == "kitti":
            full, ps, f = (32, 32, 16), 2, 16
            m = ns.unet3d_kitti.UNet3D(5, nn.BatchNorm3d, full, f, ps, context_prior=True, cascade_cls=True,
                                       occluded_cls=True).eval()
            x = torch.randn(1, f, 16, 16, 8)
        else:
            full, f = (12, 8, 12), 16
            m = ns.unet3d_nyu.UNet3D(5, nn.BatchNorm3d, f, full, context_prior=True, cascade_cls=False).eval()
            x = torch.randn(1, f, 12, 8, 12)
    synth.randomize_bn_(m)
    return m, x


def unet2d(ns):
    torch.manual_seed(0)
    with _quiet():
        m = ns.unet2d.UNet2D.build(out_feature=16, use_decoder=True, backbone_2d_name="tf_efficientnet_b3_ns",
                                   return_up_feats=1).eval()
    synth.randomize_bn_(m)
    return m, torch.randn(1, 3, 38, 45)


def occdepth_small(ns):
    """OccDepth ("flosp", kitti decoder with CRP + cascade) on a tiny stereo pair"""
    torch.manual_seed(0)
    full = (32, 32, 16)
    cfg = synth.occdepth_cfg(full_scene_size=full, feature=16, feature_2d_oc=16, n_classes=6,
                             backbone_2d_name="tf_efficientnet_b3_ns")
    with _quiet():
        m = ns.OccDepth.OccDepth(class_names=["c"] * 6, class_weights=torch.ones(6), full_scene_size=full,
                                 project_res=PROJECT_RES, config=cfg).eval()
    synth.randomize_bn_(m)
    H, W = 33, 49
    g = torch.Generator().manual_seed(0)
    img = torch.randn(1, 2, 3, H, W, generator=g)
    pix, fov = synth.random_indices(16 * 16 * 8, W, H, n_views=2, P=1, seed=5, margin=(10, 6))
    return m, {"img": img, "projected_pix_2": [pix], "fov_mask_2": [fov]}, cfg


def flosp_depth(ns):
    """FlospDepth (DepthNet + frustum grid + trilinear sampling + masked mean), kitti geometry, 2 cameras"""
    torch.manual_seed(0)
    conf = copy.deepcopy(ns.flosp_depth_conf_map["kitti"])
    H, W = 96, 320
    conf.update(scene_size=(64, 64, 8), project_scale=2, return_depth=True, final_dim=(H, W), output_channels=16,
                x_bound=[0, 12.8, 0.2], y_bound=[-6.4, 6.4, 0.2], z_bound=[-2, -0.4, 0.2], d_bound=[2.0, 18.0, 0.5],
                depth_net_conf=dict(in_channels=16, mid_channels=32))
    with _quiet():
        m = ns.FlospDepth(**conf).eval()
    synth.seed_weights_(m, 5)
    K, Ts = synth.kitti_calib(W, H, focal=220.0)
    cam_k = [torch.from_numpy(K).unsqueeze(0).repeat(2, 1, 1)]
    T = [torch.stack([torch.from_numpy(t) for t in Ts])]
    ida = [torch.eye(4).unsqueeze(0).repeat(2, 1, 1)]
    feat = torch.randn(1, 2, 16, H // 8, W // 8)
    return m, conf, (feat, cam_k, T, ida)


def nyu_virtual_batch(H, W, full, seed=0):
    g = torch.Generator().manual_seed(seed)
    img = torch.randn(1, 1, 3, H, W, generator=g)
    depth = torch.rand(1, 1, H, W, generator=g) * 7.5 + 0.5
    depth[0, 0, 3, 5] = 0.0          # exercises the inf -> 0 disparity rule (OccDepth.py:248)
    N = full[0] * full[1] * full[2]
    pix, fov = synth.random_indices(N, W, H, n_views=2, P=1, seed=seed + 1, margin=(8, 6))
    return {"img": img, "gt_depth": depth, "virtual_bf": [torch.tensor(51.88579 * W / 640.0)],
            "vox_origin": torch.zeros(1, 3, dtype=torch.float64), "projected_pix_1": [pix], "fov_mask_1": [fov]}


def occdepth_nyu_virtual_view(ns):
    """NYU-type path: one real view, the right view synthesised from gt_depth (generate_virtual_img)"""
    torch.manual_seed(0)
    full = (12, 8, 12)
    cfg = synth.occdepth_cfg(dataset="NYU", full_scene_size=full, project_scale=1, feature=16, feature_2d_oc=16,
                             n_classes=6, cascade_cls=False, backbone_2d_name="tf_efficientnet_b3_ns")
    with _quiet():
        m = ns.OccDepth.OccDepth(["c"] * 6, torch.ones(6), full_scene_size=full, project_res=PROJECT_RES,
                                 config=cfg).eval()
    synth.seed_weights_(m, 3)
    return m, nyu_virtual_batch(32, 64, full), cfg


def oracle_cfg(cfg):
    c = dict(cfg)
    c["project_res"] = PROJECT_RES
    return c
