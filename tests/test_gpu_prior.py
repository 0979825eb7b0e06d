"""FlospDepth occupancy-prior kernels (csrc/frustum.cu) vs float64 `F.grid_sample`.

`occd_grid_sample_prior_fwd` reads the sampling grids, so it isolates the trilinear sampler: grid coordinates on a
2^-10 lattice make `((g + 1) * size - 1) * 0.5` exact in fp32, and the float64 reference sees the same sample points.
`occd_frustum_sample_fwd` computes the grids from the camera tables `FlospDepth.camera_tables` builds; its reference
is `oracle.functional.frustum_grid` evaluated in float64.
"""
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import functional as OF
from oracle import synth

import gpu_cases as G

pytestmark = pytest.mark.gpu

TOL_GIVEN = 1e-5          # absolute: the inputs are probabilities, the sample points are exact


def _lib():
    from occdepth_b200 import _lib as L
    return L


def prior_ref(depth, grids, mean_mode):
    """depth float64 [V, Dn, h, w]; grids float64 [V, X, Y, Z, 3] -> [X, Y, Z] as oracle/functional.py:478-484"""
    V = depth.shape[0]
    feats, masks = [], []
    for v in range(V):
        vol = depth[v][None, None]
        g = grids[v][None]
        feats.append(F.grid_sample(vol, g, mode="bilinear", padding_mode="zeros", align_corners=False)[0, 0])
        masks.append(F.grid_sample(torch.ones_like(vol), g, mode="bilinear", padding_mode="zeros",
                                   align_corners=False)[0, 0])
    if V == 1:
        return feats[0]
    agg = sum(feats)
    if mean_mode:
        m = sum(masks)
        agg = torch.where(m > 0, agg / m, agg)
    return agg


def probabilities(V, Dn, h, w, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(V, Dn, h, w, generator=g).mul(2).softmax(1)


def lattice_grids(V, X, Y, Z, seed):
    """[V, X, Y, Z, 3] on the 2^-10 lattice in [-1.3, 1.3], with the edge cases at the first voxels"""
    g = torch.Generator().manual_seed(seed)
    gr = torch.randint(-1331, 1332, (V, X * Y * Z, 3), generator=g).double() / 1024
    q = 1.0 / 1024
    special = [(1, 1, 1), (-1, -1, -1),                          # exactly the outer texel edges
               (1 + 4 * q, 0.25, 0.5), (0.125, -1 - 3 * q, 0),     # less than half a texel outside: partial mask
               (0, 0.5, -1 - 5 * q),
               (-2, -2, -2),                                       # the non-finite sentinel in every view: msum == 0
               (5, -7, 3),                                         # far outside
               (1, -1, 1)]
    for n, xyz in enumerate(special[:X * Y * Z]):
        gr[:, n] = torch.tensor(xyz, dtype=torch.float64)
    if X * Y * Z > len(special) and V > 1:
        gr[0, len(special)] = -2                                   # outside in one view only
    return gr.reshape(V, X, Y, Z, 3)


def run_given(depth, grids, mean_mode, perm_xzy=0):
    V, Dn, h, w = depth.shape
    X, Y, Z = grids.shape[1:4]
    d = depth.float().cuda().contiguous()
    gdev = grids.float().reshape(V, -1, 3).cuda().contiguous()
    out = torch.full((X * Y * Z,), float("nan"), device="cuda")
    L = _lib()
    rc = L.lib().occd_grid_sample_prior_fwd(d.data_ptr(), gdev.data_ptr(), V, Dn, h, w, X, Y, Z, mean_mode,
                                            out.data_ptr(), perm_xzy, L.stream_ptr())
    L.check(rc, "occd_grid_sample_prior_fwd")
    torch.cuda.synchronize()
    return out.cpu()


GIVEN = [  # V, Dn, h, w, X, Y, Z   (N = X*Y*Z, none a multiple of 256)
    (1, 8, 12, 20, 7, 9, 5),
    (2, 2, 1, 1, 5, 3, 17),
    (3, 5, 1, 9, 4, 4, 4),
    (2, 2, 6, 1, 3, 11, 13),
    (3, 8, 12, 20, 7, 9, 5),
    (2, 16, 24, 40, 9, 30, 11),
]


@pytest.mark.parametrize("mean_mode", [1, 0], ids=["mean", "sum"])
@pytest.mark.parametrize("V,Dn,h,w,X,Y,Z", GIVEN)
def test_grid_sample_prior_vs_float64(V, Dn, h, w, X, Y, Z, mean_mode):
    depth = probabilities(V, Dn, h, w, seed=V * 100 + Dn)
    grids = lattice_grids(V, X, Y, Z, seed=X * Y * Z)
    # the lattice points map to exact fp32 texel coordinates
    g32 = grids.float().double()
    assert torch.equal(g32, grids)
    want = prior_ref(depth.double(), grids, mean_mode).reshape(-1)
    got = run_given(depth, grids, mean_mode).double()
    err = float((got - want).abs().max())
    G.record("grid_sample_prior[V%d,Dn%d,%dx%d,N%d]" % (V, Dn, h, w, X * Y * Z), "mean" if mean_mode else "sum",
             err=err)
    assert err <= TOL_GIVEN, err
    if mean_mode and V > 1:
        assert float(got[5]) == 0.0                       # every view outside: mask sum 0 -> 0, not NaN


def test_grid_sample_prior_perm_xzy_is_an_index_permutation():
    V, Dn, h, w, X, Y, Z = 3, 8, 12, 20, 7, 9, 5
    depth = probabilities(V, Dn, h, w, seed=1)
    grids = lattice_grids(V, X, Y, Z, seed=2)
    plain = run_given(depth, grids, 1, perm_xzy=0).view(X, Y, Z)
    perm = run_given(depth, grids, 1, perm_xzy=1).view(X, Z, Y)
    assert torch.equal(perm, plain.permute(0, 2, 1))


# ---------------------------------------------------------------------------------------------------------------
# computed grids
def _flosp(H, W):
    from occdepth_b200.models.flosp_depth import FlospDepth
    from occdepth_b200.models.flosp_depth import flosp_depth_conf_map
    import copy
    conf = copy.deepcopy(flosp_depth_conf_map["kitti"])
    # the grid starts 3.2 m behind the cameras and reaches far to the sides: voxels behind the camera, outside the
    # image and in front of the camera but nearer than dmin (the sqrt of a negative bin index) are all present
    conf.update(scene_size=(80, 64, 16), project_scale=2, return_depth=True, final_dim=(H, W), output_channels=16,
                x_bound=[-3.2, 12.8, 0.2], y_bound=[-6.4, 6.4, 0.2], z_bound=[-2, 1.2, 0.2], d_bound=[2.0, 18.0, 0.5],
                depth_net_conf=dict(in_channels=16, mid_channels=32))
    return FlospDepth(**conf), conf


def _yawed(T, angle, shift):
    c, s = math.cos(angle), math.sin(angle)
    R = torch.tensor([[c, 0, s, 0], [0, 1, 0, 0], [-s, 0, c, 0], [0, 0, 0, 1]], dtype=torch.float64)  # about camera y
    out = R @ T.double()
    out[:3, 3] += torch.tensor(shift, dtype=torch.float64)
    return out.float()


def test_frustum_sample_vs_float64():
    """sum mode over two cameras.  Zero-padded trilinear sampling is continuous in the sampling coordinate, so the
    difference from the float64 reference is bounded by the fp32 error of the computed coordinate times the largest
    texel-to-texel change of the probabilities (< 1).  Voxels within 0.1 m of an image plane are left out: there the
    perspective division 1/z amplifies the fp32 rounding of z without bound, and the reference itself is only as
    accurate as its own float32 arithmetic.  (Mean mode divides by mask sums that can be arbitrarily small at the
    volume's slivers; the given-grid cases check that arithmetic on exact sample points.)"""
    H, W = 96, 320
    m, conf = _flosp(H, W)
    K, Ts = synth.kitti_calib(W, H, focal=220.0)
    T = torch.stack([torch.from_numpy(Ts[0]), _yawed(torch.from_numpy(Ts[1]), 0.3, (0.4, 0.1, -0.5))])
    cam_k = torch.from_numpy(K).unsqueeze(0).repeat(2, 1, 1)
    ida = torch.eye(4).unsqueeze(0).repeat(2, 1, 1)
    ida[1, 0, 0], ida[1, 0, 3], ida[1, 1, 1], ida[1, 1, 3] = 0.75, 12.0, 0.75, -6.0    # a scaled, shifted crop
    cams, _, vn = m.camera_tables([cam_k], [T], [ida], None, 2)
    X, Y, Z = vn
    Dn = m.depth_channels
    h, w = H // 8, W // 8
    d0, d1 = conf["d_bound"][0], conf["d_bound"][1]
    depth = probabilities(2, Dn, h, w, seed=4)
    # float64 reference
    bounds = [conf["x_bound"], conf["y_bound"], conf["z_bound"]]
    pc_min = torch.tensor([b[0] for b in bounds], dtype=torch.float64)
    pc_max = torch.tensor([b[1] for b in bounds], dtype=torch.float64)
    grids, near = [], torch.zeros(X, Y, Z, dtype=torch.bool)
    beyond = torch.zeros(X, Y, Z, dtype=torch.bool)
    for v in range(2):
        K4 = torch.eye(4, dtype=torch.float64)
        K4[:3, :3] = cam_k[v]
        grids.append(OF.frustum_grid(vn, pc_min, pc_max, T[v].double(), K4, ida[v].double(), (H, W), Dn, d0, d1)[0])
        # camera-frame depth of every voxel centre
        vs = (pc_max - pc_min) / torch.tensor(vn, dtype=torch.float64)
        i, j, k = torch.meshgrid(*[torch.arange(n, dtype=torch.float64) for n in vn], indexing="ij")
        pts = pc_min + (torch.stack([i, j, k], -1) + 0.5) * vs
        z = pts @ T[v].double()[2, :3] + T[v].double()[2, 3]
        near |= z.abs() < 0.1
        beyond |= z < 0
    grids = torch.stack(grids)
    want = prior_ref(depth.double(), grids, 0)
    d = depth.cuda()
    out = torch.full((X * Y * Z,), float("nan"), device="cuda")
    L = _lib()
    cams_d = cams[0].cuda().contiguous()
    rc = L.lib().occd_frustum_sample_fwd(d.data_ptr(), cams_d.data_ptr(), 2, Dn, h, w, X, Y, Z, float(W), float(H),
                                         float(d0), float(d1), 0, out.data_ptr(), 0, L.stream_ptr())
    L.check(rc, "occd_frustum_sample_fwd")
    torch.cuda.synchronize()
    got = out.cpu().double().view(X, Y, Z)
    keep = ~near
    # the poses produce every branch: behind the camera, nearer than dmin, outside the image, inside
    nz = grids[..., 2]
    assert bool(beyond.any()) and bool((nz == -2).any())
    assert bool(((grids[..., 0].abs() > 1.2) & (nz > -1) & (nz < 1)).any())
    assert float((want > 0).double().mean()) > 0.1
    assert 0 < int(near.sum()) < near.numel() // 10
    err = float((got - want)[keep].abs().max())
    G.record("frustum_sample[sum]", "fp32", err=err, excluded=int(near.sum()))
    # bound: 2x the value measured on B200 (see the docstring for why it is small and why the near plane is excluded)
    assert err <= 2e-4, err


def test_prior_kernels_reject_single_depth_bin():
    L = _lib()
    d = torch.rand(1, 1, 4, 4, device="cuda")
    cams = torch.zeros(40, device="cuda")
    grids = torch.zeros(8, 3, device="cuda")
    out = torch.zeros(8, device="cuda")
    rc = L.lib().occd_frustum_sample_fwd(d.data_ptr(), cams.data_ptr(), 1, 1, 4, 4, 2, 2, 2, 32.0, 32.0, 1.0, 9.0, 0,
                                         out.data_ptr(), 0, L.stream_ptr())
    assert rc != 0 and b"occd_frustum_sample_fwd" in L.lib().occd_last_error()
    rc = L.lib().occd_grid_sample_prior_fwd(d.data_ptr(), grids.data_ptr(), 1, 1, 4, 4, 2, 2, 2, 1, out.data_ptr(), 0,
                                            L.stream_ptr())
    assert rc != 0 and b"occd_grid_sample_prior_fwd" in L.lib().occd_last_error()
    torch.cuda.synchronize()
    assert float(out.abs().max()) == 0
