"""Plain-PyTorch fp32 CPU restatement of the OccDepth forward hot path (TEST INFRASTRUCTURE ONLY).

State-dict driven and functional: every function takes the reference's `state_dict` (same key names as the
reference modules / released checkpoints) plus a key prefix, so that the same random weights can be fed
to the reference (here), to this oracle (here and on the GPU box) and to the CUDA path.
Each function cites the reference file:line it follows.  Pinned by tests/test_oracle_vs_reference.py.
"""
import math

import torch
import torch.nn.functional as F


# --------------------------------------------------------------------------------------------------
# helpers
def _bn(sd, p, x, eps=1e-5):
    """eval-mode BatchNorm (running stats), nn.BatchNorm{2,3}d default eps unless given."""
    return F.batch_norm(x, sd[p + ".running_mean"], sd[p + ".running_var"], sd[p + ".weight"], sd[p + ".bias"],
                        False, 0.0, eps)


def _conv3d(sd, p, x, stride=1, padding=0, dilation=1):
    return F.conv3d(x, sd[p + ".weight"], sd.get(p + ".bias"), stride, padding, dilation)


def _conv2d(sd, p, x, stride=1, padding=0, dilation=1, groups=1):
    return F.conv2d(x, sd[p + ".weight"], sd.get(p + ".bias"), stride, padding, dilation, groups)


# --------------------------------------------------------------------------------------------------
# A3: SFA lift -- occdepth/models/SFA.py:12-106
def sfa(x2d, projected_pix, fov_mask, scene_size, dataset, project_scale):
    """x2d (V,C,h,w) f32; projected_pix (V,N,P,2) int64 (x,y); fov_mask (V,N,P) bool -> (C,X,Y,Z)."""
    V, C, h, w = x2d.shape
    N = projected_pix.shape[1]
    feats, masks = [], []
    for v in range(V):
        src = x2d[v].reshape(C, h * w)
        x, y = projected_pix[v, :, :, 0], projected_pix[v, :, :, 1]            # SFA.py:21
        idx = (y * w + x).long()
        fov = fov_mask[v]
        idx = torch.where(fov, idx, torch.zeros_like(idx))
        g = src[:, idx.reshape(-1)].reshape(C, N, -1)                          # gather, SFA.py:28-30
        g = g * fov.unsqueeze(0).to(src.dtype)                                 # zero column for ~fov, :19-27
        cnt = fov.sum(1)                                                       # SFA.py:31
        f = g.sum(2) / cnt.unsqueeze(0)                                        # float / int64, SFA.py:32
        f = torch.where(torch.isnan(f), torch.zeros_like(f), f)                # 0/0 -> 0, SFA.py:34-38
        feats.append(f)
        masks.append((cnt > 0).to(src.dtype))                                  # SFA.py:33,39-41
    if V > 1:
        out = torch.zeros(C, N, dtype=x2d.dtype, device=x2d.device)
        for i in range(V):
            for j in range(i + 1, V):
                wij = masks[i] * masks[j]                                      # SFA.py:53-55
                cos = F.cosine_similarity(feats[i], feats[j], 0) * wij         # SFA.py:70
                wi = cos + (masks[i] > masks[j]).to(cos.dtype)                 # SFA.py:56-71
                wj = cos + (masks[j] > masks[i]).to(cos.dtype)
                out = out + (wi * feats[i] + wj * feats[j])                    # SFA.py:80-83
        out = out / (V * (V - 1))                                              # SFA.py:84-87
    else:
        out = feats[0]                                                         # SFA.py:88
    S = [s // project_scale for s in scene_size]
    if dataset == "NYU":                                                       # SFA.py:90-97
        return out.reshape(C, S[0], S[2], S[1]).permute(0, 1, 3, 2)
    return out.reshape(C, S[0], S[1], S[2])                                    # SFA.py:98-104


def lift_flosp(x_rgb, projected_pix, fov_mask, project_res, scene_size, dataset, project_scale):
    """OccDepth._forward_2d_to_3d, "flosp" branch (OccDepth.py:264-298) for ONE batch item.
    x_rgb: list over views of dict "1_s" -> (C,h,w)."""
    x3d = None
    for s in project_res:
        s = int(s)
        x2d = torch.stack([xv["1_%d" % s] for xv in x_rgb], 0)
        t = sfa(x2d, projected_pix // s, fov_mask, scene_size, dataset, project_scale)   # OccDepth.py:284-295
        x3d = t if x3d is None else x3d + t
    return x3d


# --------------------------------------------------------------------------------------------------
# A6: Bottleneck3D -- occdepth/models/DDR.py:35-139
def bottleneck3d(sd, p, x, stride=1, dilation=(1, 1, 1), downsample=False):
    d = dilation
    out1 = F.relu(_bn(sd, p + ".bn1", _conv3d(sd, p + ".conv1", x)))                                     # :114
    out2 = _bn(sd, p + ".bn2", _conv3d(sd, p + ".conv2", out1, (1, 1, stride), (0, 0, d[0]), (1, 1, d[0])))
    out3 = _bn(sd, p + ".bn3", _conv3d(sd, p + ".conv3", F.relu(out2), (1, stride, 1), (0, d[1], 0), (1, d[1], 1)))
    if stride != 1:                                                                                       # :119-120
        t = F.avg_pool3d(out2, (1, stride, 1), (1, stride, 1))
        out2 = _bn(sd, p + ".downsample2.2", _conv3d(sd, p + ".downsample2.1", t))
    out3 = out3 + out2                                                                                    # :121
    out4 = _bn(sd, p + ".bn4", _conv3d(sd, p + ".conv4", F.relu(out3), (stride, 1, 1), (d[2], 0, 0), (d[2], 1, 1)))
    if stride != 1:                                                                                       # :125-127
        out2 = _bn(sd, p + ".downsample3.2",
                   _conv3d(sd, p + ".downsample3.1", F.avg_pool3d(out2, (stride, 1, 1), (stride, 1, 1))))
        out3 = _bn(sd, p + ".downsample4.2",
                   _conv3d(sd, p + ".downsample4.1", F.avg_pool3d(out3, (stride, 1, 1), (stride, 1, 1))))
    out4 = out4 + out2 + out3                                                                             # :128
    out5 = _bn(sd, p + ".bn5", _conv3d(sd, p + ".conv5", F.relu(out4)))                                   # :130-131
    residual = x
    if downsample:                                                             # modules.py:329-339 (Downsample)
        residual = _bn(sd, p + ".downsample.2", _conv3d(sd, p + ".downsample.1", F.avg_pool3d(x, 2, 2)))
    return F.relu(out5 + residual)                                                                        # :136-139


def process(sd, p, x, dilations=(1, 2, 3)):
    """modules.py:258-275"""
    for i, dl in enumerate(dilations):
        x = bottleneck3d(sd, "%s.main.%d" % (p, i), x, 1, (dl, dl, dl))
    return x


def downsample(sd, p, x):
    """modules.py:320-344"""
    return bottleneck3d(sd, p + ".main", x, stride=2, downsample=True)


def upsample(sd, p, x):
    """modules.py:278-296: ConvTranspose3d(k3,s2,p1,op1) + BN + ReLU"""
    y = F.conv_transpose3d(x, sd[p + ".main.0.weight"], sd[p + ".main.0.bias"], 2, 1, 1, 1, 1)
    return F.relu(_bn(sd, p + ".main.1", y))


def convblock3d(sd, p, x, stride=1):
    """modules.py:299-317: ConvTranspose3d(k3,stride,p1,op0) + BN + ReLU"""
    y = F.conv_transpose3d(x, sd[p + ".main.0.weight"], sd[p + ".main.0.bias"], stride, 1, 0, 1, 1)
    return F.relu(_bn(sd, p + ".main.1", y))


def aspp_body(sd, p, x, dilations=(1, 2, 3)):
    """the ASPP block shared by modules.py:41-48 (ASPP) and the heads (:98-102, :163-166)"""
    y = None
    for i, dl in enumerate(dilations):
        t = F.relu(_bn(sd, "%s.bn1.%d" % (p, i), _conv3d(sd, "%s.conv1.%d" % (p, i), x, 1, dl, dl)))
        t = _bn(sd, "%s.bn2.%d" % (p, i), _conv3d(sd, "%s.conv2.%d" % (p, i), t, 1, dl, dl))
        y = t if y is None else y + t
    return F.relu(y + x)


def seg_head(sd, p, x):
    """SegmentationHead.forward modules.py:94-106"""
    x = F.relu(_conv3d(sd, p + ".conv0", x, 1, 1))
    x = aspp_body(sd, p, x)
    return _conv3d(sd, p + ".conv_classes", x, 1, 1)


def seg_head_cascade(sd, p, x):
    """SegmentationHeadCascadeCLS.forward modules.py:158-175"""
    x = F.relu(_conv3d(sd, p + ".conv0", x, 1, 1))
    x = aspp_body(sd, p, x)
    x_occ = _conv3d(sd, p + ".occ_classes", x, 1, 1)
    x = torch.cat([x, F.softmax(x_occ, 1)], 1)
    return _conv3d(sd, p + ".conv_classes", x, 1, 1), x_occ


def seg_head_occluded(sd, p, x):
    """SegmentationHeadOccludedCLS.forward modules.py:222-235"""
    x = F.relu(_conv3d(sd, p + ".conv0", x, 1, 1))
    x = aspp_body(sd, p, x)
    return _conv3d(sd, p + ".occ_classes", x, 1, 1)


# --------------------------------------------------------------------------------------------------
# A8: CPMegaVoxels -- occdepth/models/CRP3D.py:54-97
def cp_mega_voxels(sd, p, x, size, n_relations=4):
    bs = x.shape[0]
    flat = size[0] * size[1] * size[2]
    x_agg = aspp_body(sd, p + ".aspp", x)                                                  # :58
    pad = tuple((s + 1) % 2 for s in size)                                                 # :20
    ctx = _conv3d(sd, p + ".mega_context.0", x_agg, 2, pad)                                # :61
    cfeat = ctx.shape[1]
    ctx = ctx.reshape(bs, cfeat, -1).permute(0, 2, 1)                                      # :62-63
    logits, rels = [], []
    for r in range(n_relations):
        lg = _conv3d(sd, "%s.context_prior_logits.%d.0" % (p, r), x_agg)                   # :71
        lg = lg.reshape(bs, -1, flat)                                                      # :72-74
        logits.append(lg.unsqueeze(1))
        rels.append(torch.bmm(torch.sigmoid(lg.permute(0, 2, 1)), ctx))                    # :77-81
    xc = torch.cat(rels, 2).permute(0, 2, 1).reshape(bs, -1, size[0], size[1], size[2])    # :84-88
    y = torch.cat([x, xc], 1)                                                              # :90
    y = _conv3d(sd, p + ".resize.0", y)                                                    # :91 (1x1x1, no bias)
    y = process(sd, p + ".resize.1", y, dilations=(1,))
    return {"P_logits": torch.cat(logits, 1), "x": y}                                      # :93-97


# --------------------------------------------------------------------------------------------------
# A7: UNet3D -- unet3d_kitti.py:89-126, unet3d_nyu.py:79-110
def unet3d_kitti(sd, p, x3d, full_scene_size, project_scale, context_prior=True, cascade_cls=False,
                 occluded_cls=False, infer_mode=False):
    res = {}
    size_l1 = tuple(int(s / project_scale) for s in full_scene_size)
    size_l3 = tuple(s // 4 for s in size_l1)
    x_l1 = x3d
    x_l2 = downsample(sd, p + ".process_l1.1", process(sd, p + ".process_l1.0", x_l1))
    x_l3 = downsample(sd, p + ".process_l2.1", process(sd, p + ".process_l2.0", x_l2))
    if context_prior:
        ret = cp_mega_voxels(sd, p + ".CP_mega_voxels", x_l3, size_l3)
        x_l3 = ret["x"]
        res.update(ret)
    up_l2 = upsample(sd, p + ".up_13_l2", x_l3) + x_l2
    up_l1 = upsample(sd, p + ".up_12_l1", up_l2) + x_l1
    if project_scale == 1:
        up_full = convblock3d(sd, p + ".up_l1_lfull", up_l1)
    else:
        up_full = upsample(sd, p + ".up_l1_lfull", up_l1)
    if not infer_mode:
        res["x3d_l1"], res["x3d_l2"], res["x3d_l3"] = up_l1, up_l2, x_l3
    if cascade_cls:
        ssc, occ = seg_head_cascade(sd, p + ".ssc_head", up_full)
        res["ssc_logit"] = ssc
        if not infer_mode:
            res["occ_logit"] = occ
    else:
        res["ssc_logit"] = seg_head(sd, p + ".ssc_head", up_full)
    if occluded_cls:
        o = seg_head_occluded(sd, p + ".occluded_head", up_full)
        if not infer_mode:
            res["occluded_logit"] = o
    return res


def unet3d_nyu(sd, p, x3d, full_scene_size, n_relations=4, context_prior=True, cascade_cls=False,
               infer_mode=False):
    res = {}
    size_1_16 = tuple(int(math.ceil(i / 4)) for i in full_scene_size)
    x_1_4 = x3d
    x_1_8 = downsample(sd, p + ".process_1_4.1", process(sd, p + ".process_1_4.0", x_1_4))
    x_1_16 = downsample(sd, p + ".process_1_8.1", process(sd, p + ".process_1_8.0", x_1_8))
    if context_prior:
        ret = cp_mega_voxels(sd, p + ".CP_mega_voxels", x_1_16, size_1_16, n_relations)
        x_1_16 = ret["x"]
        res.update(ret)
    up_1_8 = upsample(sd, p + ".up_1_16_1_8", x_1_16) + x_1_8
    up_1_4 = upsample(sd, p + ".up_1_8_1_4", up_1_8) + x_1_4
    if not infer_mode:
        res["x3d_l1"], res["x3d_l2"], res["x3d_l3"] = up_1_4, up_1_8, x_1_16
    if cascade_cls:
        ssc, occ = seg_head_cascade(sd, p + ".ssc_head_1_4", up_1_4)
        res["ssc_logit"] = ssc
        if not infer_mode:
            res["occ_logit"] = occ
    else:
        res["ssc_logit"] = seg_head(sd, p + ".ssc_head_1_4", up_1_4)
    return res


# --------------------------------------------------------------------------------------------------
# A2a: EfficientNet encoder as iterated by Encoder.forward (unet2d.py:188-196); geffnet names
def _same_pad(i, k, s):
    return max((math.ceil(i / s) - 1) * s + (k - 1) + 1 - i, 0)


def _conv2d_tf(sd, p, x, k, stride, groups=1):
    if stride == 1:
        return _conv2d(sd, p, x, 1, (k - 1) // 2, 1, groups)
    ph, pw = _same_pad(x.shape[-2], k, stride), _same_pad(x.shape[-1], k, stride)
    x = F.pad(x, [pw // 2, pw - pw // 2, ph // 2, ph - ph // 2])
    return _conv2d(sd, p, x, stride, 0, 1, groups)


def _se(sd, p, x):
    s = x.mean((2, 3), keepdim=True)
    s = _conv2d(sd, p + ".conv_expand", F.silu(_conv2d(sd, p + ".conv_reduce", s)))
    return x * torch.sigmoid(s)


def effnet_features(sd, p, x, name):
    """returns the reference's `features` list (unet2d.py:189-196): [x, conv_stem, bn1, act1, blocks[0..6],
    conv_head, bn2, act2, global_pool(=Identity), classifier(=Identity)]"""
    from .effnet import block_specs, BN_EPS
    stem, specs, head = block_specs(name)
    feats = [x]
    feats.append(_conv2d_tf(sd, p + ".conv_stem", feats[-1], 3, 2))
    feats.append(_bn(sd, p + ".bn1", feats[-1], BN_EPS))
    feats.append(F.silu(feats[-1]))
    y = feats[-1]
    counters = {}
    for (si, typ, cin, cout, k, stride, e, se) in specs:
        bi = counters.get(si, 0)
        counters[si] = bi + 1
        bp = "%s.blocks.%d.%d" % (p, si, bi)
        inp = y
        if typ == "ds":
            y = F.silu(_bn(sd, bp + ".bn1", _conv2d_tf(sd, bp + ".conv_dw", y, k, stride, cin), BN_EPS))
            y = _se(sd, bp + ".se", y)
            y = _bn(sd, bp + ".bn2", _conv2d(sd, bp + ".conv_pw", y), BN_EPS)
        else:
            mid = cin * e
            y = F.silu(_bn(sd, bp + ".bn1", _conv2d(sd, bp + ".conv_pw", y), BN_EPS))
            y = F.silu(_bn(sd, bp + ".bn2", _conv2d_tf(sd, bp + ".conv_dw", y, k, stride, mid), BN_EPS))
            y = _se(sd, bp + ".se", y)
            y = _bn(sd, bp + ".bn3", _conv2d(sd, bp + ".conv_pwl", y), BN_EPS)
        if stride == 1 and cin == cout:
            y = y + inp
        if bi + 1 == sum(1 for s in specs if s[0] == si):
            feats.append(y)
    feats.append(_conv2d(sd, p + ".conv_head", y))
    feats.append(_bn(sd, p + ".bn2", feats[-1], BN_EPS))
    feats.append(F.silu(feats[-1]))
    feats.append(feats[-1])  # global_pool = Identity (unet2d.py:245)
    feats.append(feats[-1])  # classifier = Identity (unet2d.py:246)
    return feats


# A2b: DecoderBN -- unet2d.py:137-165, UpSampleBN :24-46
def _upsample_bn(sd, p, x, skip):
    up = F.interpolate(x, size=(skip.shape[2], skip.shape[3]), mode="bilinear", align_corners=True)
    f = torch.cat([up, skip], 1)
    f = F.leaky_relu(_bn(sd, p + "._net.1", _conv2d(sd, p + "._net.0", f, 1, 1)), 0.01)
    return F.leaky_relu(_bn(sd, p + "._net.4", _conv2d(sd, p + "._net.3", f, 1, 1)), 0.01)


def decoder_bn(sd, p, features, return_up_feats=1):
    b0, b1, b2, b3, b4 = features[4], features[5], features[6], features[8], features[11]
    x_d0 = _conv2d(sd, p + ".conv2", b4, 1, 1)               # 1x1 conv WITH padding=1 (unet2d.py:65-67)
    res = {}
    x16 = _upsample_bn(sd, p + ".up16", x_d0, b3)
    res["1_16"] = _conv2d(sd, p + ".resize_output_1_16", x16)
    if return_up_feats <= 8:
        x8 = _upsample_bn(sd, p + ".up8", x16, b2)
        res["1_8"] = _conv2d(sd, p + ".resize_output_1_8", x8)
    if return_up_feats <= 4:
        x4 = _upsample_bn(sd, p + ".up4", x8, b1)
        res["1_4"] = _conv2d(sd, p + ".resize_output_1_4", x4)
    if return_up_feats <= 2:
        x2 = _upsample_bn(sd, p + ".up2", x4, b0)
        res["1_2"] = _conv2d(sd, p + ".resize_output_1_2", x2)
    if return_up_feats <= 1:
        x1 = _upsample_bn(sd, p + ".up1", x2, features[0])
        res["1_1"] = _conv2d(sd, p + ".resize_output_1_1", x1)
    return res


def unet2d(sd, p, x, backbone="tf_efficientnet_b7_ns", return_up_feats=1):
    """UNet2D.forward unet2d.py:221-224"""
    feats = effnet_features(sd, p + ".encoder.original_model", x, backbone)
    return decoder_bn(sd, p + ".decoder", feats, return_up_feats)


# --------------------------------------------------------------------------------------------------
# A2c: virtual right view -- OccDepth.generate_virtual_img (OccDepth.py:233-260)
def virtual_view(x, depth, scale_2d, bf):
    """x (B,C,h,w) left features; depth (B,1,H,W); returns the disparity-shifted right-view features."""
    n, c, h, w = x.shape
    dm = F.interpolate(depth, size=(h, w), mode="bilinear", align_corners=False)        # :240-244
    dx = (bf / int(scale_2d)) / dm                                                      # :246-247
    dx = torch.where(torch.isinf(dx), torch.zeros_like(dx), dx).to(x.dtype)
    hd = torch.arange(-1, 1, 2 / h, device=x.device)                                    # :249-250 (corner coords)
    wd = torch.arange(-1, 1, 2 / w, device=x.device)
    my, mx = torch.meshgrid(hd, wd, indexing="ij")
    grid = torch.stack((mx, my), 2).unsqueeze(0).repeat(n, 1, 1, 1).to(x.dtype)
    grid[..., 0] = grid[..., 0] + (dx * 2 / w)[0]                                       # item 0's disparity, :255-257
    return F.grid_sample(x, grid, mode="bilinear", padding_mode="border", align_corners=False)


# --------------------------------------------------------------------------------------------------
# A1: OccDepth.forward, "flosp" transform (OccDepth.py:344-376)
def occdepth_forward(sd, batch, cfg):
    """cfg: dict(dataset, full_scene_size, project_scale, project_res, backbone_2d_name, return_up_feats,
    context_prior, cascade_cls, occluded_cls, n_relations, infer_mode)"""
    img = batch["img"]
    bs, n_views = img.shape[:2]
    x_rgb = [unet2d(sd, "net_rgb", img[:, v], cfg["backbone_2d_name"], cfg["return_up_feats"])
             for v in range(n_views)]                                           # process_rgbs :208-219
    if n_views == 1 and "gt_depth" in batch:                                    # process_rgbs :221-229
        bf = batch["virtual_bf"][0]
        x_rgb.append({"1_" + str(s): virtual_view(x_rgb[0]["1_" + str(s)], batch["gt_depth"], s, bf)
                      for s in cfg["project_res"]})
        n_views = 2
    ps = cfg["project_scale"]
    x3ds = []
    for i in range(bs):
        xv = [{k: t[i] for k, t in xr.items()} for xr in x_rgb]
        x3ds.append(lift_flosp(xv, batch["projected_pix_%d" % ps][i], batch["fov_mask_%d" % ps][i],
                               cfg["project_res"], cfg["full_scene_size"], cfg["dataset"], ps))
    x3d = torch.stack(x3ds)
    extra = {}
    if cfg.get("trans_2d_to_3d", "flosp") == "flosp_depth":                      # OccDepth.py:299-339
        conf = cfg["flosp_depth_conf"]
        layer = "1_%d" % conf["downsample_factor"]
        nv = 1 if cfg["dataset"] == "NYU" else n_views
        img_feat = torch.stack([x_rgb[j][layer] for j in range(nv)], 1)
        vox_origin = batch.get("vox_origin") if cfg["dataset"] == "NYU" else None
        prior, depth_pred = flosp_depth(sd, "flosp_depth", img_feat, batch["cam_k"], batch["T_velo_2_cam"],
                                        batch["ida_mats"], conf, vox_origin)
        if cfg["dataset"] == "NYU":
            prior = prior.permute(0, 1, 2, 4, 3)
        x3d = x3d * prior * 100
        if cfg.get("with_depth_gt", False):
            extra["depth_pred"] = depth_pred
    ctx = cfg["context_prior"] and not cfg.get("infer_mode", False)             # OccDepth.py:82-84
    if cfg["dataset"] == "NYU":
        out = unet3d_nyu(sd, "net_3d_decoder", x3d, cfg["full_scene_size"], cfg.get("n_relations", 4), ctx,
                         cfg["cascade_cls"], cfg.get("infer_mode", False))
    else:
        out = unet3d_kitti(sd, "net_3d_decoder", x3d, cfg["full_scene_size"], ps, ctx, cfg["cascade_cls"],
                           cfg.get("occluded_cls", False), cfg.get("infer_mode", False))
    out.update(extra)
    return out


# --------------------------------------------------------------------------------------------------
# A4/A5: FlospDepth -- flosp_depth.py:201-257 (DepthNet), :456-608 (forward); f2v/frustum_grid_generator.py:70-152
def depth_net(sd, p, x, cam_k4):
    """x (BV, C, h, w); cam_k4 (BV, 4, 4) intrinsics.  flosp_depth.py:232-257"""
    inv = torch.inverse(cam_k4)
    sps = torch.norm(torch.stack([inv[..., 0, 0], inv[..., 1, 1]], dim=-1), dim=-1).reshape(-1, 1) * 1000.0
    x = F.relu(_bn(sd, p + ".reduce_conv.1", _conv2d(sd, p + ".reduce_conv.0", x, 1, 1)))
    h = F.linear(F.relu(F.linear(sps, sd[p + ".mlp.fc1.weight"], sd[p + ".mlp.fc1.bias"])),
                 sd[p + ".mlp.fc2.weight"], sd[p + ".mlp.fc2.bias"])[..., None, None]
    g = _conv2d(sd, p + ".se.conv_expand", F.relu(_conv2d(sd, p + ".se.conv_reduce", h)))
    x = x * torch.sigmoid(g)
    for i in range(3):
        q = "%s.depth_conv.%d" % (p, i)
        y = F.relu(_bn(sd, q + ".bn1", _conv2d(sd, q + ".conv1", x, 1, 1)))
        x = F.relu(_bn(sd, q + ".bn2", _conv2d(sd, q + ".conv2", y, 1, 1)) + x)
    return _conv2d(sd, p + ".depth_pred", x)


def frustum_grid(grid_size, pc_min, pc_max, lidar_to_cam, cam_k4, ida, image_hw, num_bins, dmin, dmax):
    """frustum_grid_generator.py:20-152 for one camera: -> (1, X, Y, Z, 3) normalised sampling grid."""
    X, Y, Z = grid_size
    dt = lidar_to_cam.dtype                      # float32 as in the reference; float64 for kernel-level tests
    vs = (pc_max - pc_min) / torch.tensor([X, Y, Z], dtype=dt)
    i, j, k = torch.meshgrid(torch.arange(X, dtype=dt), torch.arange(Y, dtype=dt),
                             torch.arange(Z, dtype=dt), indexing="ij")
    vox = torch.stack([i, j, k], -1) + 0.5                                       # :31-42
    G = torch.eye(4, dtype=dt)
    G[0, 0], G[1, 1], G[2, 2] = vs
    G[:3, 3] = pc_min
    trans = lidar_to_cam @ G                                                     # :95
    ph = F.pad(vox, [0, 1], value=1.0) @ trans.t()                                # kornia.transform_points :102
    z = ph[..., 3:]
    cam = ph[..., :3] * torch.where(z.abs() > 1e-8, 1.0 / (z + 1e-8), torch.ones_like(z))
    I_C = cam_k4[:3, :]
    pt = F.pad(cam, [0, 1], value=1.0) @ I_C.t()                                  # transform_utils.py:16-21
    zz = pt[..., 2:]
    img = pt[..., :2] * torch.where(zz.abs() > 1e-8, 1.0 / (zz + 1e-8), torch.ones_like(zz))
    depth = pt[..., 2] - I_C[2, 3]                                                # :24
    bin_size = 2 * (dmax - dmin) / (num_bins * (1 + num_bins))                    # depth_utils.py:24-26
    idx = -0.5 + 0.5 * torch.sqrt(1 + 8 * (depth - dmin) / bin_size)
    fg = torch.cat([img, idx.unsqueeze(-1)], -1)
    fh = F.pad(fg, [0, 1], value=1.0) @ ida.t()                                   # :113-114
    w = fh[..., 3:]
    fg = fh[..., :3] * torch.where(w.abs() > 1e-8, 1.0 / (w + 1e-8), torch.ones_like(w))
    shape = torch.tensor([float(image_hw[1]), float(image_hw[0]), float(num_bins)], dtype=dt)   # flipped [D,H,W], :139-145
    fg = fg / (shape - 1) * 2 - 1
    fg[~torch.isfinite(fg)] = -2                                                  # :148-150
    return fg.unsqueeze(0)


def flosp_depth(sd, p, img_feat, cam_k, T_velo_2_cam, ida_mats, conf, vox_origin=None):
    """FlospDepth.forward (flosp_depth.py:456-608).  img_feat (B, n_cams, C, h, w); returns (B,1,X,Y,Z), depth."""
    B, V, C, h, w = img_feat.shape
    ps = conf["project_scale"]
    if vox_origin is not None:                                                    # :466-518 (NYU)
        o = [float(vox_origin[0][k]) for k in range(3)]
        bounds = [[o[0], o[0] + 4.8, 0.08], [o[1], o[1] + 4.8, 0.08], [o[2], o[2] + 2.88, 0.08]]
    else:
        bounds = [conf["x_bound"], conf["y_bound"], conf["z_bound"]]
    vn = [int((b[1] - b[0]) / b[2] / ps) for b in bounds]
    pc_min = torch.tensor([b[0] for b in bounds], dtype=torch.float32)
    pc_max = torch.tensor([b[1] for b in bounds], dtype=torch.float32)
    d_bound = conf["d_bound"]
    Dn = int((d_bound[1] - d_bound[0]) / d_bound[2])
    K4 = torch.zeros(B, V, 4, 4)
    K4[:, :, :3, :3] = torch.stack(cam_k).to(torch.float32)
    K4[:, :, 3, 3] = 1
    T = torch.stack(T_velo_2_cam).to(torch.float32)
    ida = torch.stack(ida_mats)
    logits = depth_net(sd, p + ".depth_net.0", img_feat.reshape(B * V, C, h, w), K4.reshape(B * V, 4, 4))
    depth = logits.softmax(1).reshape(B, V, 1, Dn, h, w)                          # :548-559
    feats, masks = [], []
    for v in range(V):
        grids = torch.cat([frustum_grid(vn, pc_min, pc_max, T[b, v], K4[b, v], ida[b, v], conf["final_dim"], Dn,
                                        d_bound[0], d_bound[1]) for b in range(B)], 0)
        feats.append(F.grid_sample(depth[:, v], grids, mode="bilinear", padding_mode="zeros", align_corners=False))
        masks.append(F.grid_sample(torch.ones_like(depth[:, v]), grids, mode="bilinear", padding_mode="zeros",
                                   align_corners=False))
    if V == 1:
        agg = feats[0]
    else:
        agg = sum(feats)
        if conf.get("agg_voxel_mode", "mean") == "mean":
            m = sum(masks)
            agg = torch.where(m > 0, agg / m, agg)                                # :594-602
    return agg, depth.squeeze(2)
