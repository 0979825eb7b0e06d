"""The drop-in boundary: every module of occdepth_b200.models must expose exactly the reference's state_dict keys
and shapes (released checkpoints are loaded with strict=True, scripts/eval.py:65-70).  The reference's layouts were
recorded by oracle/gen_golden.py in tests/golden/state_dict_keys.json.xz."""
import copy
import json
import lzma
import os

import pytest
import torch

from oracle import gen_golden, synth
from oracle.reference_cases import PROJECT_RES

with lzma.open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "state_dict_keys.json.xz"),
               "rt") as _f:
    GOLD = json.load(_f)
CONFIGS = {name: (args, kw) for name, args, kw in gen_golden.state_dict_configs()}


def _same(a, name):
    """`a` has the recorded layout, key order included, and a checkpoint of that layout loads into it"""
    sa, want = a.state_dict(), GOLD[name]
    assert [k for k, _, _ in want] == list(sa.keys())
    ckpt = {}
    for k, shape, dtype in want:
        assert list(sa[k].shape) == shape and str(sa[k].dtype) == dtype, k
        ckpt[k] = torch.zeros(shape, dtype=getattr(torch, dtype.split(".")[-1]))
    a.load_state_dict(ckpt, strict=True)      # and a reference checkpoint loads
    return len(sa)


def test_unet3d_keys():
    from occdepth_b200.models import unet3d_kitti, unet3d_nyu
    args, kw = CONFIGS["unet3d_kitti[full]"]
    assert _same(unet3d_kitti.UNet3D(*args, **kw), "unet3d_kitti[full]") > 500
    args, kw = CONFIGS["unet3d_nyu[full]"]
    assert _same(unet3d_nyu.UNet3D(*args, **kw), "unet3d_nyu[full]") > 500
    args, kw = CONFIGS["unet3d_kitti[project_scale_1]"]      # project_scale 1 -> Convblock3d
    assert _same(unet3d_kitti.UNet3D(*args, **kw), "unet3d_kitti[project_scale_1]") > 300


@pytest.mark.parametrize("backbone", ["tf_efficientnet_b3_ns", "tf_efficientnet_b4_ns", "tf_efficientnet_b5_ns",
                                      "tf_efficientnet_b7_ns"])
def test_unet2d_keys(backbone):
    from occdepth_b200.models import unet2d
    name = "unet2d[%s]" % backbone
    assert _same(unet2d.UNet2D.build(**CONFIGS[name][1]), name) > 600


def test_flosp_depth_keys():
    from occdepth_b200.models.flosp_depth import FlospDepth, flosp_depth_conf_map
    assert json.loads(json.dumps(flosp_depth_conf_map)) == GOLD["flosp_depth_conf_map"]
    for ds in ("kitti", "NYU"):
        name = "flosp_depth[%s]" % ds
        kw = CONFIGS[name][1]
        c = copy.deepcopy(flosp_depth_conf_map[kw["dataset"]])
        c.update(kw["update"])
        assert _same(FlospDepth(**c), name) == 56


@pytest.mark.parametrize("variant", ["kitti_flosp", "kitti_flosp_depth", "nyu_flosp"])
def test_occdepth_keys(variant):
    from occdepth_b200.models.OccDepth import OccDepth
    import occdepth_b200.models.flosp_depth.flosp_depth as mfd
    name = "occdepth[%s]" % variant
    cfg = synth.Cfg(CONFIGS[name][1])
    saved = copy.deepcopy(mfd.flosp_depth_conf_map)
    try:
        n = _same(OccDepth(["c"] * cfg.n_classes, torch.ones(cfg.n_classes), full_scene_size=cfg.full_scene_size,
                           project_res=PROJECT_RES, config=cfg), name)
    finally:       # OccDepth mutates the module-level conf dicts in place, as the reference does (OccDepth.py:183-198)
        for k in mfd.flosp_depth_conf_map:
            mfd.flosp_depth_conf_map[k].clear()
            mfd.flosp_depth_conf_map[k].update(saved[k])
    assert n > 1800
