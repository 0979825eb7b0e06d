"""Pins oracle/functional.py against the UNMODIFIED reference modules (CPU fp32, seeded weights).

The reference outputs were recorded by oracle/gen_golden.py on the cases of oracle/reference_cases.py and are
stored in tests/golden/reference_outputs.pt: whole tensors up to 1024 elements, else 512 elements at fixed indices
(reference_cases.sample_index) plus the sum of the whole tensor; the numba vox2pix as sha256 digests of its arrays.
"""
import os

import pytest
import torch

from oracle import functional as OF
from oracle import reference_cases as RC

GOLD = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_outputs.pt"))
TOL = dict(rtol=1e-4, atol=1e-5)


@pytest.fixture(scope="module")
def ns():
    return RC.product_modules()


def _close(a, want, **kw):
    """`a` against a packed reference output: elementwise allclose on the stored elements, and on the whole tensor
    the bound on the sum that elementwise allclose implies"""
    tol = dict(TOL)
    tol.update(kw)
    assert tuple(a.shape) == want["shape"], (a.shape, want["shape"])
    flat = a.detach().flatten()
    got = flat[RC.sample_index(flat.numel())] if want["sampled"] else flat
    assert torch.allclose(got, want["values"], **tol), float((got - want["values"]).abs().max())
    err = abs(float(flat.double().sum()) - want["sum"])
    assert err <= tol["atol"] * flat.numel() + tol["rtol"] * want["abs_sum"], err


def _unpack(want):
    assert not want["sampled"]
    return want["values"].view(want["shape"])


def _same_weights(case, *modules):
    """this package's modules built from the case's seed hold the weights the reference modules held"""
    got, want = RC.state_sum(*modules), GOLD[case]["state_sum"]
    assert all(abs(g - w) <= 1e-12 * abs(w) for g, w in zip(got, want)), (got, want)     # float64 summation order


@pytest.mark.parametrize("dataset,V,P", RC.SFA_CASES)
def test_sfa(dataset, V, P):
    c = RC.sfa(dataset, V, P)
    got = OF.sfa(c["x2d"], c["pix"], c["fov"], c["scene"], dataset, c["ps"])
    _close(got, GOLD["sfa[%s-%d-%d]" % (dataset, V, P)]["out"], rtol=1e-5, atol=1e-6)


def test_bottleneck_process_downsample(ns):
    proc, down, up, x = RC.bottleneck(ns)
    _same_weights("bottleneck", proc, down, up)
    gold = GOLD["bottleneck"]
    with torch.no_grad():
        _close(OF.process({"p." + k: v for k, v in proc.state_dict().items()}, "p", x), gold["process"])
        _close(OF.downsample({"p." + k: v for k, v in down.state_dict().items()}, "p", x), gold["downsample"])
        y = _unpack(gold["downsample"])        # the reference's Downsample output feeds its Upsample
        _close(OF.upsample({"p." + k: v for k, v in up.state_dict().items()}, "p", y), gold["upsample"])


@pytest.mark.parametrize("which", ["kitti", "nyu"])
def test_unet3d(ns, which):
    m, x = RC.unet3d(ns, which)
    case = "unet3d[%s]" % which
    _same_weights(case, m)
    sd = {"n." + k: v for k, v in m.state_dict().items()}
    with torch.no_grad():
        if which == "kitti":
            got = OF.unet3d_kitti(sd, "n", x, (32, 32, 16), 2, True, True, True)
        else:
            got = OF.unet3d_nyu(sd, "n", x, (12, 8, 12), 4, True, False)
    want = GOLD[case]["out"]
    assert set(got.keys()) == set(want.keys())
    for k in want:
        _close(got[k], want[k], rtol=1e-3, atol=1e-4)


def test_unet2d(ns):
    m, x = RC.unet2d(ns)
    _same_weights("unet2d", m)
    sd = {"net_rgb." + k: v for k, v in m.state_dict().items()}
    with torch.no_grad():
        got = OF.unet2d(sd, "net_rgb", x, "tf_efficientnet_b3_ns", 1)
    want = GOLD["unet2d"]["out"]
    assert set(got.keys()) == set(want.keys())
    for k in want:
        _close(got[k], want[k], rtol=1e-3, atol=1e-4)


def test_occdepth_forward_small(ns):
    """whole OccDepth.forward ("flosp", kitti decoder with CRP + cascade) on a tiny stereo pair."""
    m, batch, cfg = RC.occdepth_small(ns)
    _same_weights("occdepth_small", m)
    with torch.no_grad():
        got = OF.occdepth_forward(m.state_dict(), batch, RC.oracle_cfg(cfg))
    want = GOLD["occdepth_small"]["out"]
    assert set(got.keys()) == set(want.keys())
    for k in want:
        _close(got[k], want[k], rtol=2e-3, atol=2e-4)


def test_flosp_depth(ns):
    """FlospDepth (DepthNet + frustum grid + trilinear sampling + masked mean), kitti geometry, 2 cameras"""
    m, conf, (feat, cam_k, T, ida) = RC.flosp_depth(ns)
    _same_weights("flosp_depth", m)
    gold = GOLD["flosp_depth"]
    with torch.no_grad():
        got, got_d = OF.flosp_depth({"f." + k: v for k, v in m.state_dict().items()}, "f", feat, cam_k, T, ida, conf)
    assert gold["covered"] > 0.2     # the frustum actually covers part of the grid
    _close(got_d, gold["depth"], rtol=1e-4, atol=1e-6)
    _close(got, gold["out"], rtol=1e-3, atol=1e-5)


def test_occdepth_forward_nyu_virtual_view(ns):
    """NYU-type path: one real view, the right view synthesised from gt_depth (generate_virtual_img)"""
    m, batch, cfg = RC.occdepth_nyu_virtual_view(ns)
    _same_weights("occdepth_nyu_virtual_view", m)
    with torch.no_grad():
        got = OF.occdepth_forward(m.state_dict(), batch, RC.oracle_cfg(cfg))
    want = GOLD["occdepth_nyu_virtual_view"]["out"]
    assert set(got.keys()) == set(want.keys())
    for k in want:
        _close(got[k], want[k], rtol=2e-3, atol=2e-4)


@pytest.mark.parametrize("pattern_id", RC.VOX2PIX_PATTERNS)
def test_vox2pix_against_the_numba_reference(pattern_id):
    """oracle/projection.py vs occdepth.data.utils.helpers.vox2pix itself (numba-compiled), bit for bit"""
    from oracle import gen_golden, projection
    for name, E, K, org, vs, W, H, scene, _ in gen_golden.vox2pix_cases():
        want = GOLD["vox2pix[%s-%d]" % (name, pattern_id)]
        got = projection.vox2pix(E, K, org, vs, W, H, scene, pattern_id)
        assert [gen_golden.array_digest(g) for g in got] == want, name
