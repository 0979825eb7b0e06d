"""Generates tests/golden/* by running the UNMODIFIED reference (imported through oracle/ref_import.py, which finds
its source tree through OCCDEPTH_REFERENCE) on seeded inputs and weights:  python -m oracle.gen_golden

Each fixture stores the inputs (or the seed that regenerates them), the seed of `synth.seed_weights_`, and the
reference outputs (fp16-safe small tensors kept as fp32).
"""
import copy
import hashlib
import json
import lzma
import os

import numpy as np
import torch
import torch.nn as nn

from . import ref_import, synth

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def sfa_cases():
    return [("kitti", 2, 1, 16), ("NYU", 2, 1, 16), ("kitti", 1, 1, 8), ("kitti", 2, 5, 8), ("kitti", 3, 1, 8)]


def gen_sfa(ref):
    out = {}
    scene, ps, h, w = (12, 10, 8), 2, 9, 17
    N = 6 * 5 * 4
    for i, (ds, V, P, C) in enumerate(sfa_cases()):
        g = torch.Generator().manual_seed(100 + i)
        x2d = torch.randn(V, C, h, w, generator=g)
        pix, fov = synth.random_indices(N, w, h, n_views=V, P=P, seed=200 + i, margin=(4, 3))
        y = ref.SFA.SFA(scene, ds, ps)(x2d, pix.clone(), fov.clone()).contiguous()
        out["case%d" % i] = dict(dataset=ds, x2d=x2d, pix=pix, fov=fov, out=y, scene=scene, ps=ps)
    torch.save(out, os.path.join(OUT, "sfa.pt"))


def gen_unet3d(ref):
    with ref_import.quiet():
        mk = ref.unet3d_kitti.UNet3D(5, nn.BatchNorm3d, (32, 32, 16), 16, 2, context_prior=True, cascade_cls=True,
                                     occluded_cls=True).eval()
        mn = ref.unet3d_nyu.UNet3D(5, nn.BatchNorm3d, 16, (12, 8, 12), context_prior=True, cascade_cls=False).eval()
    synth.seed_weights_(mk, 11)
    synth.seed_weights_(mn, 12)
    g = torch.Generator().manual_seed(3)
    xk = torch.randn(1, 16, 16, 16, 8, generator=g)
    xn = torch.randn(1, 16, 12, 8, 12, generator=g)
    with torch.no_grad():
        ok, on = mk({"x3d": xk}), mn({"x3d": xn})
    keep = ("ssc_logit", "occ_logit", "occluded_logit", "P_logits")
    torch.save(dict(kitti=dict(x=xk, seed=11, out={k: v for k, v in ok.items() if k in keep}),
                    nyu=dict(x=xn, seed=12, out={k: v for k, v in on.items() if k in keep})),
               os.path.join(OUT, "unet3d.pt"))


def gen_occdepth(ref):
    full = (32, 32, 16)
    cfg = synth.occdepth_cfg(full_scene_size=full, feature=16, feature_2d_oc=16, n_classes=6,
                             backbone_2d_name="tf_efficientnet_b3_ns")
    with ref_import.quiet():
        m = ref.OccDepth.OccDepth(["c"] * 6, torch.ones(6), full_scene_size=full, project_res=["1", "2", "4", "8"],
                                  config=cfg).eval()
    synth.seed_weights_(m, 21)
    H, W = 33, 49
    g = torch.Generator().manual_seed(0)
    img = torch.randn(1, 2, 3, H, W, generator=g)
    pix, fov = synth.random_indices(16 * 16 * 8, W, H, n_views=2, P=1, seed=5, margin=(10, 6))
    with torch.no_grad():
        out = m({"img": img, "projected_pix_2": [pix], "fov_mask_2": [fov]})
        feats = m.net_rgb(img[:, 0])
    torch.save(dict(img=img, pix=pix, fov=fov, seed=21, cfg=dict(cfg), ssc_logit=out["ssc_logit"],
                    occ_logit=out["occ_logit"], feat_1_8=feats["1_8"], feat_1_1_mean=feats["1_1"].mean((2, 3))),
               os.path.join(OUT, "occdepth_small.pt"))


def vox2pix_cases():
    """(name, cam_E, cam_k, vox_origin, voxel_size, img_W, img_H, scene_size, pattern_id): a KITTI-like rig with a
    slightly rotated pose (so every term of the pose matrix matters), an NYU-like one, and a camera INSIDE the volume
    (voxels behind it and one column of centres in the camera plane: z <= 0, division by zero)"""
    import math
    import numpy as np

    def rot(ax, a):
        c, s = math.cos(a), math.sin(a)
        R = np.eye(3)
        i, j = [(1, 2), (0, 2), (0, 1)][ax]
        R[i, i] = c; R[j, j] = c; R[i, j] = -s; R[j, i] = s
        return R
    base = np.array([[0, -1, 0], [0, 0, -1], [1, 0, 0.0]])
    E1 = np.eye(4)
    E1[:3, :3] = rot(0, 0.03) @ rot(1, -0.02) @ rot(2, 0.01) @ base
    E1[:3, 3] = [0.011, -0.083, -0.271]
    K1 = np.array([[707.0912, 0, 601.8873], [0, 707.0912, 183.1104], [0, 0, 1.0]])
    E2 = np.eye(4)
    E2[:3, :3] = rot(0, -0.4) @ rot(2, 0.7)
    E2[:3, 3] = [0.3, -0.2, 1.1]
    K2 = np.array([[518.8579, 0, 320.0], [0, 518.8579, 240.0], [0, 0, 1.0]])
    E3 = np.eye(4)
    E3[:3, :3] = base
    E3[:3, 3] = [0.0, 0.0, -0.75]         # cam z = lidar x - 0.75: the centres at x = 0.75 lie exactly in the camera plane
    return [("kitti_p0", E1, K1, np.array([0, -6.4, -2.0]), 0.4, 1220, 370, (12.8, 12.8, 3.2), 0),
            ("kitti_p3", E1, K1, np.array([0, -6.4, -2.0]), 0.8, 1220, 370, (12.8, 12.8, 3.2), 3),
            ("nyu_p8", E2.astype(np.float32), K2, np.array([-1.2, -1.0, 0.1]), 0.16, 640, 480, (2.4, 2.4, 1.44), 8),
            ("plane_p1", E3, K1, np.array([0.0, -2.0, -1.0]), 0.5, 1220, 370, (4.0, 4.0, 2.0), 1)]


def gen_vox2pix():
    helpers = ref_import.data_helpers()
    out = {}
    for name, E, K, org, vs, W, H, scene, pid in vox2pix_cases():
        pix, fov, z = helpers.vox2pix(E, K, org, vs, W, H, scene, pid)
        if np.array_equal(pix.astype(np.int16), pix):      # stored as int16 where that is lossless (file size)
            pix = pix.astype(np.int16)
        out[name] = dict(cam_E=torch.from_numpy(E.copy()), cam_k=torch.from_numpy(K.copy()),
                         vox_origin=torch.from_numpy(org.copy()), voxel_size=vs, img_W=W, img_H=H,
                         scene_size=scene, pattern_id=pid, pix=torch.from_numpy(pix), fov=torch.from_numpy(fov),
                         pix_z=torch.from_numpy(z))
    torch.save(out, os.path.join(OUT, "vox2pix.pt"))


def pack(t, full_max=1024):
    """a reference output for the golden file: all of it up to `full_max` elements, else its elements at
    reference_cases.sample_index; with the float64 sum and absolute sum of the whole tensor"""
    from .reference_cases import sample_index
    t = t.detach().float().contiguous()
    flat = t.flatten()
    d = dict(shape=tuple(t.shape), sum=float(t.double().sum()), abs_sum=float(t.double().abs().sum()),
             sampled=flat.numel() > full_max)
    d["values"] = flat[sample_index(flat.numel())].clone() if d["sampled"] else flat.clone()
    return d


def array_digest(a):
    """sha256 of an array's dtype, shape and bytes (NaNs canonicalised): bit-exact comparisons without the array"""
    a = np.array(a)
    if a.dtype.kind == "f":
        a[np.isnan(a)] = np.nan
    h = hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode())
    h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def gen_reference_outputs():
    """what tests/test_oracle_vs_reference.py compares the oracle with: the reference modules' outputs on the seeded
    cases of oracle/reference_cases.py, and digests of the numba vox2pix for every case and pattern"""
    from . import reference_cases as RC
    ns = RC.reference_modules()
    out = {}
    with torch.no_grad():
        for ds, V, P in RC.SFA_CASES:
            c = RC.sfa(ds, V, P)
            y = ns.SFA.SFA(c["scene"], ds, c["ps"])(c["x2d"], c["pix"].clone(), c["fov"].clone())
            out["sfa[%s-%d-%d]" % (ds, V, P)] = dict(out=pack(y.contiguous()))
        proc, down, up, x = RC.bottleneck(ns)
        y = down(x)
        out["bottleneck"] = dict(state_sum=RC.state_sum(proc, down, up), process=pack(proc(x)),
                                 downsample=pack(y, full_max=y.numel()), upsample=pack(up(y)))
        for which in ("kitti", "nyu"):
            m, x = RC.unet3d(ns, which)
            out["unet3d[%s]" % which] = dict(state_sum=RC.state_sum(m),
                                             out={k: pack(v) for k, v in m({"x3d": x}).items()})
        m, x = RC.unet2d(ns)
        out["unet2d"] = dict(state_sum=RC.state_sum(m), out={k: pack(v) for k, v in m(x).items()})
        m, batch, _ = RC.occdepth_small(ns)
        out["occdepth_small"] = dict(state_sum=RC.state_sum(m), out={k: pack(v) for k, v in m(batch).items()})
        m, _, args = RC.flosp_depth(ns)
        y, d = m(*args, None)
        out["flosp_depth"] = dict(state_sum=RC.state_sum(m), out=pack(y), depth=pack(d),
                                  covered=float((y > 0).float().mean()))
        m, batch, _ = RC.occdepth_nyu_virtual_view(ns)
        out["occdepth_nyu_virtual_view"] = dict(state_sum=RC.state_sum(m),
                                                out={k: pack(v) for k, v in m(batch).items()})
    helpers = ref_import.data_helpers()
    for pid in RC.VOX2PIX_PATTERNS:
        for name, E, K, org, vs, W, H, scene, _ in vox2pix_cases():
            out["vox2pix[%s-%d]" % (name, pid)] = [array_digest(a) for a in helpers.vox2pix(E, K, org, vs, W, H,
                                                                                              scene, pid)]
    torch.save(out, os.path.join(OUT, "reference_outputs.pt"))


def gen_state_dict_keys():
    """state_dict layout (key, shape, dtype) of the reference modules in the configurations of
    tests/test_state_dict_compat.py, and the reference's FlospDepth configuration map"""
    from . import reference_cases as RC
    ns = RC.reference_modules()

    def layout(m):
        return [[k, list(v.shape), str(v.dtype)] for k, v in m.state_dict().items()]
    out = {}
    with ref_import.quiet():
        for name, args, kw in state_dict_configs():
            if name.startswith("unet3d_kitti"):
                out[name] = layout(ns.unet3d_kitti.UNet3D(*args, **kw))
            elif name.startswith("unet3d_nyu"):
                out[name] = layout(ns.unet3d_nyu.UNet3D(*args, **kw))
            elif name.startswith("unet2d"):
                out[name] = layout(ns.unet2d.UNet2D.build(**kw))
            elif name.startswith("flosp_depth"):
                c = copy.deepcopy(ns.flosp_depth_conf_map[kw["dataset"]])
                c.update(kw["update"])
                out[name] = layout(ns.FlospDepth(**c))
            else:
                cfg = synth.Cfg(kw)
                saved = copy.deepcopy(ns.flosp_depth_conf_map)
                try:
                    out[name] = layout(ns.OccDepth.OccDepth(["c"] * cfg.n_classes, torch.ones(cfg.n_classes),
                                                            full_scene_size=cfg.full_scene_size,
                                                            project_res=RC.PROJECT_RES, config=cfg))
                finally:       # the reference mutates the module-level conf dicts in place (OccDepth.py:183-198)
                    for k, v in saved.items():
                        ns.flosp_depth_conf_map[k].clear()
                        ns.flosp_depth_conf_map[k].update(v)
    out["flosp_depth_conf_map"] = json.loads(json.dumps(ns.flosp_depth_conf_map))
    with lzma.open(os.path.join(OUT, "state_dict_keys.json.xz"), "wt") as f:
        json.dump(out, f, separators=(",", ":"))


def state_dict_configs():
    """(name, args, kwargs) of every module configuration whose state_dict layout tests/test_state_dict_compat.py
    checks; OccDepth entries carry their config dict as kwargs"""
    k3 = dict(context_prior=True, cascade_cls=True, occluded_cls=True)
    cfgs = [("unet3d_kitti[full]", (20, nn.BatchNorm3d, (256, 256, 32), 64, 2), k3),
            ("unet3d_nyu[full]", (12, nn.BatchNorm3d, 200, (60, 36, 60)), {}),
            ("unet3d_kitti[project_scale_1]", (20, nn.BatchNorm3d, (128, 128, 16), 32, 1), {})]
    for b in ("tf_efficientnet_b3_ns", "tf_efficientnet_b4_ns", "tf_efficientnet_b5_ns", "tf_efficientnet_b7_ns"):
        cfgs.append(("unet2d[%s]" % b, (), dict(out_feature=64, use_decoder=True, backbone_2d_name=b,
                                                 return_up_feats=1)))
    for ds, scene, ps in (("kitti", (256, 256, 32), 2), ("NYU", (60, 36, 60), 1)):
        cfgs.append(("flosp_depth[%s]" % ds, (), dict(dataset=ds, update=dict(scene_size=scene, project_scale=ps,
                                                                              return_depth=False))))
    cfgs.append(("occdepth[kitti_flosp]", (), dict(synth.occdepth_cfg(trans_2d_to_3d="flosp"))))
    cfgs.append(("occdepth[kitti_flosp_depth]", (), dict(synth.occdepth_cfg(trans_2d_to_3d="flosp_depth"))))
    cfgs.append(("occdepth[nyu_flosp]", (), dict(synth.occdepth_cfg(
        dataset="NYU", full_scene_size=(60, 36, 60), project_scale=1, feature=200, feature_2d_oc=200, n_classes=12,
        cascade_cls=False))))
    return cfgs


def main():
    os.makedirs(OUT, exist_ok=True)
    ref = ref_import.modules()
    torch.manual_seed(0)
    gen_sfa(ref)
    gen_unet3d(ref)
    gen_occdepth(ref)
    gen_vox2pix()
    gen_reference_outputs()
    gen_state_dict_keys()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
