"""Stereo-SFA lift -- drop-in for the reference `occdepth/models/SFA.py` (class SFA, :5-106).

`SFA(scene_size, dataset, project_scale).forward(x2d[V,C,h,w] f32, projected_pix[V,N,P,2] int64,
fov_mask[V,N,P] bool) -> [C,X,Y,Z] f32`, computed by the fused sm_100a kernel `occd_sfa_lift_fwd`.
`lift_multiscale` is the fused fast path used by OccDepth.forward (all 2D scales, both views, one launch,
channels-last bf16 in and out).
"""
import ctypes as C

import torch
import torch.nn as nn

from .. import _lib
from ..engine import CL, require_cuda


def _fill_common(p, pix, fov, n_views, Cch):
    V, N, P, two = pix.shape
    assert two == 2 and V == n_views and tuple(fov.shape) == (V, N, P)
    p.n_views, p.C = V, Cch
    p.pix, p.fov = pix.data_ptr(), fov.data_ptr()
    p.N, p.P = N, P


def _nyu_perm(p, dataset, scene_size, project_scale):
    if dataset == "NYU":
        p.perm_nyu = 1
        p.S1 = scene_size[1] // project_scale
        p.S2 = scene_size[2] // project_scale
    elif dataset == "kitti":
        p.perm_nyu = 0
    else:
        raise NotImplementedError("dataset is not supported: {}".format(dataset))


class SFA(nn.Module):
    def __init__(self, scene_size, dataset, project_scale):
        super().__init__()
        self.scene_size = scene_size
        self.dataset = dataset
        self.project_scale = project_scale

    def forward(self, x2d, projected_pix, fov_mask):
        require_cuda(x2d, "SFA.forward")
        n_views, c, h, w = x2d.shape
        dev = x2d.device
        if c % 4 != 0:
            raise RuntimeError("SFA: channel count must be a multiple of 4")
        pix = projected_pix.to(device=dev, dtype=torch.int64).contiguous()
        fov = fov_mask.to(device=dev, dtype=torch.bool).contiguous()
        # NCHW fp32 -> channels-last fp32 (the kernel gathers one contiguous C-vector per pixel).  A plain copy, not
        # occd_planar_to_cl: that one rounds to TF32, and this module returns the reference's exact fp32 lift
        feat = x2d.float().permute(0, 2, 3, 1).contiguous()
        L = _lib.lib()
        st = _lib.stream_ptr()
        S = [s // self.project_scale for s in self.scene_size]
        N = pix.shape[1]
        if N != S[0] * S[1] * S[2]:
            raise RuntimeError("SFA: projected_pix has %d voxels, scene has %d" % (N, S[0] * S[1] * S[2]))
        out = torch.empty(c, S[0], S[1], S[2], dtype=torch.float32, device=dev)
        p = _lib.SfaParams()
        p.feat[0], p.h[0], p.w[0], p.div[0] = feat.data_ptr(), h, w, 1
        p.n_scales, p.feat_dtype = 1, _lib.DTYPE_F32
        _fill_common(p, pix, fov, n_views, c)
        p.out, p.out_mode, p.out_cstride = out.data_ptr(), _lib.SFA_OUT_F32_PLANAR, c
        _nyu_perm(p, self.dataset, self.scene_size, self.project_scale)
        _lib.check(L.occd_sfa_lift_fwd(C.byref(p), st), "occd_sfa_lift_fwd")
        return out


def lift_multiscale(feats, divs, projected_pix, fov_mask, out, dataset, scene_size, project_scale, prior=None,
                    scale_const=1.0, stream=None):
    """Fused lift over all 2D scales.  feats: list of channels-last bf16 tensors [V, h_s, w_s, C] whose views may be
    strided (e.g. a [V, B, h, w, C] buffer sliced at one batch item); out: CL with dims (1, X, Y, Z) receiving
    sum_s SFA_s (x prior x scale_const)."""
    p = _lib.SfaParams()
    V = feats[0].shape[0]
    Cch = feats[0].shape[3]
    for i, (f, dv) in enumerate(zip(feats, divs)):
        assert f.dtype == feats[0].dtype and f.shape[0] == V and f.shape[3] == Cch
        assert f[0].is_contiguous() and f.stride(3) == 1
        p.feat[i], p.h[i], p.w[i], p.div[i] = f.data_ptr(), f.shape[1], f.shape[2], int(dv)
        p.vstride[i] = f.stride(0) if V > 1 else 0
    tf32 = feats[0].dtype == torch.float32
    assert tf32 or feats[0].dtype == torch.bfloat16
    assert out.buf.dtype == feats[0].dtype
    p.n_scales, p.feat_dtype = len(feats), (_lib.DTYPE_F32 if tf32 else _lib.DTYPE_BF16)
    _fill_common(p, projected_pix, fov_mask, V, Cch)
    assert out.coff == 0 and out.C == Cch and out.spatial() == p.N
    p.out, p.out_mode, p.out_cstride = out.ptr, (_lib.SFA_OUT_TF32_CL if tf32 else _lib.SFA_OUT_BF16_CL), out.cstride
    _nyu_perm(p, dataset, scene_size, project_scale)
    if prior is not None:
        assert prior.dtype == torch.float32 and prior.numel() == p.N
        p.prior, p.scale_const = prior.data_ptr(), float(scale_const)
    _lib.check(_lib.lib().occd_sfa_lift_fwd(C.byref(p), _lib.stream_ptr() if stream is None else stream),
               "occd_sfa_lift_fwd")
    return out
