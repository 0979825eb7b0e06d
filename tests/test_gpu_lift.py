"""SFA lift kernel (`occd_sfa_lift_fwd`, csrc/sfa_lift.cu) through the C ABI vs a float64 reference.

`launch_v` -> `launch_nv` -> `launch_g` pick one of 80 kernel instantiations: {P == 1 fast kernel, general staged
kernel} x {fp32, bf16 features} x V = 1..4 x five (NV, G) lane buckets per feature type.  `CASES` is a table that
names, for every case, the instantiation those rules select; `test_case_table_covers_every_instantiation` asserts
that it reaches all 80, so a new bucket cannot go untested.  The edges (N not a multiple of a block, 1-4 scales with
power-of-two and other divisors, negative and last-row/column pixels, out-of-range flat indices, fov in no / one /
all views, zero feature vectors, strided views, the NYU permutation, the prior product) are spread over the table.

The reference is `oracle.functional.sfa` run in float64 on the same (fp32- or bf16-valued) features, summed over
scales as `lift_flosp` does, then multiplied by prior * scale_const in the output voxel order (OccDepth.py:337-339).
"""
import ctypes as C
import itertools

import pytest
import torch

from oracle import functional as OF

import gpu_cases as G

DTYPES = ("f32", "bf16")
TORCH = {"f32": torch.float32, "bf16": torch.bfloat16}
VEC = {"f32": 4, "bf16": 8}          # channels per 16-byte vector (FeatTraits<T>::VEC)
MODES = ("F32_PLANAR", "F32_CL", "TF32_CL", "BF16_CL")
# the (NV, G) lane buckets of launch_nv, in order of channel count: fp32 uses 4 vectors per lane above 16 channels,
# bf16 uses 2 above 32
BUCKETS = {"f32": ((1, 4), (4, 2), (4, 4), (4, 8), (4, 16)),
           "bf16": ((1, 4), (2, 4), (2, 8), (2, 16), (2, 32))}
BUCKET_C = {"f32": (16, 32, 64, 128, 256), "bf16": (32, 64, 128, 256, 512)}     # largest C of each bucket
ODD_C = {"f32": (12, 28, 36, 100, 200), "bf16": (24, 56, 72, 200, 264)}         # other counts in the same buckets
TOL_F32 = 1e-5            # fp32 outputs, as the SFA module tests
TOL = {"F32_PLANAR": TOL_F32, "F32_CL": TOL_F32, "TF32_CL": G.TOL["tf32"], "BF16_CL": G.TOL["bf16"]}
H0, W0 = 23, 37           # image size the pixel coordinates refer to
SENTINEL = 0xA5           # byte pattern pre-filled into every output buffer


def instantiation(dt, C_, P, fits_int32=True):
    """(kernel, NV, G) that launch_nv / launch_g select, or None when C is refused"""
    vecs = -(-C_ // VEC[dt])
    if vecs <= 4:
        return ("p1" if P == 1 and fits_int32 else "general"), 1, 4
    limits = (8, 16, 32, 64)
    if vecs > limits[-1]:
        return None
    nv, g = BUCKETS[dt][1 + next(i for i, lim in enumerate(limits) if vecs <= lim)]
    return ("p1" if P == 1 and fits_int32 else "general"), nv, g


def _build_cases():
    cases = []
    for i, (dt, V, b, kern) in enumerate(itertools.product(DTYPES, (1, 2, 3, 4), range(5), ("p1", "general"))):
        ns = 1 + i % 4
        odd_divs = ns <= 3 and (i // 4) % 2 == 1
        perm = ((5, 7, 4), (3, 4, 9))[i % 2] if i % 5 == 2 else None
        cases.append(dict(
            id="%s-V%d-b%d-%s-%d" % (dt, V, b, kern, i), dt=dt, V=V,
            C=BUCKET_C[dt][b] if i % 3 else ODD_C[dt][b],
            P=1 if kern == "p1" else 2 + (i // 2) % 2,
            N=(1000, 1, 11, 777, 300, 129)[i % 6],
            divs=((1, 3, 5) if odd_divs else (1, 2, 4, 8))[:ns],
            strided=(i // 3) % 2 == 1,
            perm=perm,
            prior=i % 3 == 1,
            mode=MODES[(i // 2) % 4],
            seed=i))
    return cases


CASES = _build_cases()


def test_case_table_covers_every_instantiation():
    want = {(dt, V, kern) + nvg for dt in DTYPES for V in (1, 2, 3, 4) for kern in ("p1", "general")
            for nvg in BUCKETS[dt]}
    assert len(want) == 80
    got = {(c["dt"], c["V"]) + instantiation(c["dt"], c["C"], c["P"]) for c in CASES}
    assert got == want, sorted(want - got)
    # every output mode with both feature types (BF16_CL with fp32 features takes the 4-wide store branch)
    assert {(c["dt"], c["mode"]) for c in CASES} == set(itertools.product(DTYPES, MODES))
    assert any(c["perm"] and c["prior"] for c in CASES) and any(c["perm"] and not c["prior"] for c in CASES)
    assert {c["divs"] for c in CASES} >= {(1, 2, 4, 8), (1, 3, 5)}
    assert any(C_ not in BUCKET_C[dt] for dt in DTYPES for C_ in {c["C"] for c in CASES if c["dt"] == dt})


# ---------------------------------------------------------------------------------------------------------------
# reference
def lift_ref(feats, divs, pix, fov, perm=None, prior=None, scale_const=1.0):
    """feats: per scale float64 [V, h, w, C]; pix [V, N, P, 2] int64 (x, y); fov [V, N, P] bool.
    -> float64 [N, C] in the kernel's output voxel order.

    A point with fov set whose flat index (y // d) * w + (x // d) falls outside [0, h*w) gathers zeros but still
    counts toward the mean and the view mask (the kernel's documented behaviour; the reference's gather would raise
    or wrap there).  It is modelled by pointing such points at an extra all-zero row appended to the feature map."""
    V, N, P, _ = pix.shape
    C_ = feats[0].shape[3]
    scene, dataset = (perm, "NYU") if perm else ((N, 1, 1), "kitti")
    out = torch.zeros(C_, N, dtype=torch.float64)
    for f, d in zip(feats, divs):
        h, w = f.shape[1:3]
        ps = pix // d                                   # floor division, as OccDepth.py:286-294
        idx = ps[..., 1] * w + ps[..., 0]
        oob = fov & ((idx < 0) | (idx >= h * w))
        ps = torch.where(oob.unsqueeze(-1), torch.tensor([0, h], dtype=torch.int64), ps)
        x2d = torch.cat([f, torch.zeros(V, 1, w, C_, dtype=f.dtype)], 1).permute(0, 3, 1, 2)
        out += OF.sfa(x2d, ps, fov, scene, dataset, 1).reshape(C_, N)
    if prior is not None:
        out = out * prior.double().unsqueeze(0) * scale_const
    return out.t()


# ---------------------------------------------------------------------------------------------------------------
# inputs and the C ABI call
def make_inputs(dt, V, C_, P, N, divs, seed):
    g = torch.Generator().manual_seed(seed)
    feats = []
    for d in divs:
        h, w = -(-H0 // d), -(-W0 // d)
        f = torch.randn(V, h, w, C_, generator=g).to(TORCH[dt])
        f[:, 0, 0] = 0                                  # a zero feature vector: the cosine's eps clamp
        feats.append(f)
    x = torch.randint(-3, W0 + 3, (V, N, P), generator=g)
    y = torch.randint(-3, H0 + 3, (V, N, P), generator=g)
    pix = torch.stack([x, y], -1)
    fov = torch.rand(V, N, P, generator=g) < 0.7
    special = [(W0 - 1, H0 - 1), (0, 0), (-1, 2), (-5, -4), (W0 - 1, 0), (0, H0 - 1)]
    for n, xy in enumerate(special[:N]):                # last row/column, the zero vector, negative coordinates
        pix[:, n, 0] = torch.tensor(xy)
        fov[:, n, 0] = True
    if N > 8:
        fov[:, 6] = False                               # in no view
        fov[:, 7] = False
        fov[0, 7, 0] = True                             # in view 0 only: the m[a] > m[b] weights
        fov[:, 8] = True                                # in every pattern point of every view: the mean
    return feats, pix, fov


def place_views(f, strided):
    """device copy of f [V, h, w, C]; strided: the views sit 2*h*w*C elements apart with NaN between them (as
    OccDepth slices a [V, B, h, w, C] buffer at one batch item).  -> (tensor view, vstride argument)"""
    V, h, w, C_ = f.shape
    if not strided:
        return f.cuda().contiguous(), 0
    buf = torch.full((V, 2, h, w, C_), float("nan"), dtype=f.dtype, device="cuda")
    view = buf[:, 1]
    view.copy_(f.cuda())
    return view, view.stride(0)


def lift_params(feats_dev, vstrides, divs, dt, pix, fov, out, mode, cstride, perm=None, prior=None, scale_const=1.0):
    from occdepth_b200 import _lib
    p = _lib.SfaParams()
    for i, (f, vs, d) in enumerate(zip(feats_dev, vstrides, divs)):
        p.feat[i], p.h[i], p.w[i], p.div[i], p.vstride[i] = f.data_ptr(), f.shape[1], f.shape[2], d, vs
    p.n_scales, p.n_views, p.C = len(feats_dev), pix.shape[0], feats_dev[0].shape[3]
    p.feat_dtype = _lib.DTYPE_F32 if dt == "f32" else _lib.DTYPE_BF16
    p.pix, p.fov, p.N, p.P = pix.data_ptr(), fov.data_ptr(), pix.shape[1], pix.shape[2]
    p.out, p.out_mode, p.out_cstride = out.data_ptr(), getattr(_lib, "SFA_OUT_" + mode), cstride
    if perm:
        p.perm_nyu, p.S1, p.S2 = 1, perm[1], perm[2]
    if prior is not None:
        p.prior, p.scale_const = prior.data_ptr(), scale_const
    return p


def call(p):
    from occdepth_b200 import _lib
    rc = _lib.lib().occd_sfa_lift_fwd(C.byref(p), _lib.stream_ptr())
    return rc, (_lib.lib().occd_last_error() or b"").decode()


def alloc_out(mode, N, C_, cstride):
    """output buffer with one guard row (voxel N, or channel C for the planar layout), every byte SENTINEL"""
    dt = torch.bfloat16 if mode == "BF16_CL" else torch.float32
    shape = (C_ + 1, N) if mode == "F32_PLANAR" else (N + 1, cstride)
    buf = torch.full(shape, SENTINEL, dtype=torch.uint8, device="cuda").repeat_interleave(
        torch.finfo(dt).bits // 8, -1)
    return buf.view(dt)


def unchanged(t):
    return bool((t.contiguous().view(torch.uint8) == SENTINEL).all())


def read_out(out, mode, N, C_):
    """-> (float64 [N, C] result, sentinel regions that must be untouched)"""
    if mode == "F32_PLANAR":
        return out[:C_].t().double().cpu(), [out[C_]]
    return out[:N, :C_].double().cpu(), [out[:, C_:], out[N]]


def run_case(dt, V, C_, P, N, divs, mode, strided=False, perm=None, with_prior=False, seed=0):
    feats, pix, fov = make_inputs(dt, V, C_, P, N, divs, seed)
    prior, sc = None, 1.0
    if with_prior:
        prior, sc = torch.rand(N, generator=torch.Generator().manual_seed(seed + 1)), 100.0
    want = lift_ref([f.double() for f in feats], divs, pix, fov, perm, prior, sc)
    placed = [place_views(f, strided) for f in feats]
    cstride = C_ + 8
    out = alloc_out(mode, N, C_, cstride)
    pix_d, fov_d = pix.cuda(), fov.cuda()
    prior_d = prior.cuda() if prior is not None else None
    p = lift_params([f for f, _ in placed], [vs for _, vs in placed], divs, dt, pix_d, fov_d, out, mode, cstride,
                    perm, prior_d, sc)
    rc, msg = call(p)
    assert rc == 0, msg
    torch.cuda.synchronize()
    got, pads = read_out(out, mode, N, C_)
    for pad in pads:
        assert unchanged(pad), "pad channels / guard row overwritten"
    if mode == "TF32_CL":
        g32 = out[:N, :C_].cpu()
        assert torch.equal(g32, G.tf32r(g32)), "TF32_CL stored a value that is not TF32"
    err = float((got - want).abs().max()) / max(1.0, float(want.abs().max()))
    return err, got, want


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c["id"] for c in CASES])
def test_lift_vs_float64(case):
    c = case
    if c["perm"]:
        S = c["perm"]
        N = S[0] * S[1] * S[2]
    else:
        N = c["N"]
    err, _, _ = run_case(c["dt"], c["V"], c["C"], c["P"], N, c["divs"], c["mode"], c["strided"], c["perm"],
                         c["prior"], c["seed"])
    G.record("sfa_lift[%s]" % c["id"], c["mode"], err=err, instantiation=list(instantiation(c["dt"], c["C"], c["P"])))
    assert err <= TOL[c["mode"]], err


@pytest.mark.gpu
def test_lift_n0_writes_nothing():
    feats, pix, fov = make_inputs("f32", 2, 32, 1, 4, (1,), 0)
    f = feats[0].cuda()
    out = alloc_out("F32_CL", 4, 32, 40)
    pix_d, fov_d = pix.cuda(), fov.cuda()
    p = lift_params([f], [0], (1,), "f32", pix_d, fov_d, out, "F32_CL", 40)
    p.N = 0
    rc, msg = call(p)
    torch.cuda.synchronize()
    assert rc == 0, msg
    assert unchanged(out)


@pytest.mark.gpu
def test_lift_int32_fallback_takes_general_kernel():
    """bf16, V = 2, views 2^30 elements apart: V * vstride does not fit 32 bits, so a P == 1 input takes the general
    kernel (sfa_fits_int32 false).  Compared with the float64 reference and with the same input at dense vstride."""
    C_, N, V = 64, 1000, 2
    assert instantiation("bf16", C_, 1, fits_int32=False)[0] == "general"
    feats, pix, fov = make_inputs("bf16", V, C_, 1, N, (1,), 7)
    f = feats[0]
    hwc = f[0].numel()
    vstride = 2 ** 30
    big = torch.empty(vstride + hwc, dtype=torch.bfloat16, device="cuda")      # ~2.1 GB, only the views are filled
    big[:hwc].copy_(f[0].reshape(-1))
    big[vstride:vstride + hwc].copy_(f[1].reshape(-1))
    view = big.as_strided(f.shape, (vstride,) + tuple(f[0].stride()))
    want = lift_ref([f.double()], (1,), pix, fov)
    pix_d, fov_d = pix.cuda(), fov.cuda()
    res = {}
    for name, fv, vs in (("far", view, vstride), ("dense", f.cuda(), 0)):
        out = alloc_out("F32_CL", N, C_, C_ + 8)
        rc, msg = call(lift_params([fv], [vs], (1,), "bf16", pix_d, fov_d, out, "F32_CL", C_ + 8))
        assert rc == 0, msg
        torch.cuda.synchronize()
        got, pads = read_out(out, "F32_CL", N, C_)
        assert all(unchanged(t) for t in pads)
        res[name] = got
    del big
    scale = max(1.0, float(want.abs().max()))
    errs = {k: float((v - want).abs().max()) / scale for k, v in res.items()}
    errs["far_vs_dense"] = float((res["far"] - res["dense"]).abs().max()) / scale
    G.record("sfa_lift[int32_fallback]", "F32_CL", **errs)
    for k, e in errs.items():
        assert e <= TOL_F32, (k, e)


@pytest.mark.gpu
def test_lift_large_pattern_count_uses_dynamic_smem_opt_in():
    """V = 4, fp32 C = 32 (G = 2), P = 5: the index staging needs 170 KB of dynamic shared memory"""
    assert 4 * 128 * 4 * 5 * 17 > 48 * 1024
    err, _, _ = run_case("f32", 4, 32, 5, 300, (1, 2), "F32_CL", seed=11)
    G.record("sfa_lift[P5_smem_opt_in]", "F32_CL", err=err)
    assert err <= TOL_F32, err


@pytest.mark.gpu
@pytest.mark.parametrize("dt,V,C_,P,what", [("f32", 2, 260, 1, "C too large"), ("bf16", 2, 520, 1, "C too large"),
                                            ("f32", 4, 32, 6, "pattern count too large")])
def test_lift_refusals(dt, V, C_, P, what):
    """refused on the host before any launch, with OCCD_ERR_UNSUPPORTED and a message"""
    N = 10
    feats, pix, fov = make_inputs(dt, V, C_, P, N, (1,), 0)
    f = feats[0].cuda()
    out = alloc_out("F32_CL", N, C_, C_ + 8)
    rc, msg = call(lift_params([f], [0], (1,), dt, pix.cuda(), fov.cuda(), out, "F32_CL", C_ + 8))
    torch.cuda.synchronize()
    assert rc == 3, (rc, msg)       # OCCD_ERR_UNSUPPORTED
    assert what in msg, msg
    assert unchanged(out)
