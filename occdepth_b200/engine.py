"""Host-side execution engine: channels-last activation buffers + planned kernel launches.

PyTorch is used for device memory and streams only; every operator is a C-ABI call into libocc_b200.so
(include/occdepth_b200.h).  A `Plan` is a static list of prepared launches over pre-allocated buffers
(weights packed once, TMA descriptors encoded once), so a forward pass is a replay -- optionally captured
into a CUDA graph.
"""
import ctypes as C
import os

import torch

from . import _lib

ACT = dict(none=_lib.ACT_NONE, relu=_lib.ACT_RELU, leaky=_lib.ACT_LEAKY, silu=_lib.ACT_SILU,
           sigmoid=_lib.ACT_SIGMOID)


def _round_up(a, b):
    return (a + b - 1) // b * b


PRECISIONS = ("tf32", "bf16")
TORCH_DTYPE = {"tf32": torch.float32, "bf16": torch.bfloat16}
LIB_DTYPE = {"tf32": _lib.DTYPE_F32, "bf16": _lib.DTYPE_BF16}


def default_precision():
    """Arithmetic mode of the planned forward (OCCDEPTH_PRECISION, default 'tf32'):

    'tf32': activations are fp32 tensors holding TF32 values, convolutions run as tcgen05 kind::tf32 with fp32
            accumulation -- the reference's precision (fp32 nn.Conv*d, which PyTorch itself executes on TF32 tensor
            cores on CUDA); this is the mode the parity tests and the bench headline use.
    'bf16': bf16 activations and operands (kind::f16), fp32 accumulation -- the throughput mode, own tolerance."""
    v = os.environ.get("OCCDEPTH_PRECISION", "tf32").lower()
    if v not in PRECISIONS:
        raise ValueError("OCCDEPTH_PRECISION must be 'tf32' or 'bf16'")
    return v


def precision_of(torch_dtype):
    return "tf32" if torch_dtype == torch.float32 else "bf16"


def round_tf32_(t):
    """fp32 tensor -> nearest TF32 value (10-bit mantissa, ties away from zero == cvt.rna.tf32.f32), in place"""
    i = t.view(torch.int32)
    i.add_(0x1000).bitwise_and_(-0x2000)
    return t


def chunk_channels(C_, esize):
    """channels per K chunk (one swizzled smem row of 32 / 64 / 128 bytes), mirrors csrc/conv.cu"""
    for rb in (32, 64, 128):
        if C_ <= rb // esize:
            return rb // esize
    return 128 // esize


def default_impl():
    """'auto' (default): halo-tile tcgen05 kernel where the shape qualifies, the x-packed per-tap kernel for
    narrow-output convs with W taps, else the per-tap tcgen05 kernel; 'tc' / 'tcx' / 'halo' / 'simt' force one
    implementation (simt = CUDA-core cross-check)."""
    v = os.environ.get("OCCDEPTH_CONV_IMPL", "auto").lower()
    if v not in ("auto", "tc", "simt", "halo", "halox", "tcx"):
        raise ValueError("OCCDEPTH_CONV_IMPL must be 'auto', 'tc', 'tcx', 'halo', 'halox' or 'simt'")
    return {"auto": None, "tc": _lib.CONV_IMPL_TC, "simt": _lib.CONV_IMPL_SIMT, "halo": _lib.CONV_IMPL_HALO,
            "halox": _lib.CONV_IMPL_HALOX, "tcx": _lib.CONV_IMPL_TCX}[v]


def halox_eligible(srcs, taps, stride, omul, out_dims, Cout_pad, weight_buf):
    """shape test mirroring plan_halox (csrc/conv.cu): stride-1 'same' conv on a grid whose innermost extent W is
    8 / 16 / 32, taps = (dz, dy) groups of dx = -d, 0, +d with dz, dy in {-d, 0, d}, one K chunk, 3*Cout_pad <= 256"""
    if len(srcs) != 1 or weight_buf is not None or len(taps) % 3 or not 3 <= len(taps) <= 27:
        return False
    if tuple(stride) != (1, 1, 1) or tuple(omul) != (1, 1, 1) or tuple(out_dims) != tuple(srcs[0].dims[1:]):
        return False
    if srcs[0].dims[3] not in (8, 16, 32) or srcs[0].C > 128 // srcs[0].esize or 3 * Cout_pad > 256:
        return False
    d = taps[2][3]
    if d < 1 or d >= srcs[0].dims[3]:
        return False
    for i in range(0, len(taps), 3):
        a, b, c = taps[i], taps[i + 1], taps[i + 2]
        if not (a[:3] == b[:3] == c[:3] and (a[3], b[3], c[3]) == (-d, 0, d)):
            return False
        if a[1] not in (-d, 0, d) or a[2] not in (-d, 0, d):
            return False
    return True


def tcx_eligible(taps, stride, Cout_pad):
    """(src, dz, dy) groups of three W taps -1, 0, +1 (what conv_taps emits for a dense 3-wide kernel), W stride 1,
    N = 3*Cout_pad <= 256, and enough output channels that the packed MMA beats three narrow ones (measured on
    B200, profiles/r02_convbench_tcx.txt: Cout 80 0.154 -> 0.102 ms; Cout 32 loses to the halo kernel)"""
    if len(taps) % 3 or 3 * Cout_pad > 256 or Cout_pad < 48 or stride[2] != 1:
        return False
    for i in range(0, len(taps), 3):
        a, b, c = taps[i], taps[i + 1], taps[i + 2]
        if not (a[:3] == b[:3] == c[:3] and (a[3], b[3], c[3]) == (-1, 0, 1)):
            return False
    return True


def halo_eligible(srcs, taps, stride, omul, out_dims, Cout_pad, weight_buf):
    """shape test mirroring plan_halo (csrc/conv.cu): stride-1 'same' conv, {-d,0,d} taps, one K chunk"""
    if len(srcs) != 1 or weight_buf is not None or len(taps) < 3 or len(taps) > 27:
        return False
    if tuple(stride) != (1, 1, 1) or tuple(omul) != (1, 1, 1) or tuple(out_dims) != tuple(srcs[0].dims[1:]):
        return False
    if srcs[0].C > 128 // srcs[0].esize or Cout_pad > 64:
        return False
    offs = {abs(o) for t in taps for o in t[1:] if o}
    return len(offs) == 1


def require_cuda(t, what):
    if not (isinstance(t, torch.Tensor) and t.is_cuda):
        raise RuntimeError("%s: occdepth_b200 runs on CUDA (sm_100a) only -- there is no CPU fallback" % what)


class CL:
    """channels-last activation (bf16, or fp32 holding TF32 values): a channel window [coff, coff+C) of a
    [B,D,H,W,cstride] buffer.

    X-slab multi-GPU partition: a buffer may carry `halo` margin planes on both sides of D; the CL then denotes the
    INTERIOR planes [d0, d0+dlen) (what this rank owns and writes) while convolutions read the margins
    (neighbour data put there by HaloExchangeOp, zeros at the global boundary).  Requires B == 1."""

    def __init__(self, buf, C_, coff=0, d0=0, dlen=None):
        assert buf.dtype in (torch.bfloat16, torch.float32) and buf.dim() == 5 and buf.is_contiguous()
        self.buf, self.C, self.coff = buf, int(C_), int(coff)
        self.d0 = int(d0)
        self.dlen = int(buf.shape[1] - 2 * d0 if dlen is None else dlen)
        assert self.coff % 8 == 0 and buf.shape[4] % 8 == 0 and self.coff + self.C <= buf.shape[4]
        assert self.d0 == 0 or buf.shape[0] == 1

    @staticmethod
    def alloc(B, D, H, W, C_, device, halo=0, precision=None):
        dt = TORCH_DTYPE[precision or default_precision()]
        buf = torch.zeros(B, D + 2 * halo, H, W, _round_up(C_, 8), dtype=dt, device=device)
        return CL(buf, C_, 0, halo, D)

    @property
    def halo(self):
        return self.d0

    @property
    def precision(self):
        return precision_of(self.buf.dtype)

    @property
    def lib_dtype(self):
        return LIB_DTYPE[self.precision]

    @property
    def esize(self):
        return self.buf.element_size()

    @property
    def dims(self):
        return (self.buf.shape[0], self.dlen, self.buf.shape[2], self.buf.shape[3])

    @property
    def cstride(self):
        return self.buf.shape[4]

    @property
    def plane_elems(self):
        return self.buf.shape[2] * self.buf.shape[3] * self.buf.shape[4]

    @property
    def ptr(self):
        """pointer to the first INTERIOR plane"""
        return self.buf.data_ptr() + self.esize * self.d0 * self.plane_elems

    @property
    def full_ptr(self):
        return self.buf.data_ptr()

    def window(self, coff, C_):
        return CL(self.buf, C_, self.coff + coff, self.d0, self.dlen)

    def spatial(self):
        return self.dlen * self.buf.shape[2] * self.buf.shape[3]

    def interior(self):
        """torch view [B, dlen, H, W, cstride] of the owned planes"""
        return self.buf[:, self.d0:self.d0 + self.dlen]

    # ---- module-boundary conversions (reference tensors are NCHW / NCDHW fp32) ----
    @staticmethod
    def from_planar(x, out=None, precision=None):
        """x: fp32 [B,C,H,W] or [B,C,D,H,W] (CUDA) -> CL."""
        require_cuda(x, "CL.from_planar")
        x = x.contiguous().float()
        if x.dim() == 4:
            B, C_, H, W = x.shape
            D = 1
        else:
            B, C_, D, H, W = x.shape
        if out is None:
            out = CL.alloc(B, D, H, W, C_, x.device, precision=precision)
        assert out.coff == 0 and out.C == C_
        S = D * H * W
        rc = _lib.lib().occd_planar_to_cl(x.data_ptr(), out.ptr, out.lib_dtype, B, C_, S, out.cstride,
                                          _lib.stream_ptr())
        _lib.check(rc, "occd_planar_to_cl")
        return out

    def to_planar(self, squeeze_d=False):
        """-> fp32 [B,C,D,H,W] (or [B,C,H,W] when squeeze_d)."""
        B, D, H, W = self.dims
        out = torch.empty(B, self.C, D, H, W, dtype=torch.float32, device=self.buf.device)
        S = D * H * W
        rc = _lib.lib().occd_cl_to_planar(self.ptr + self.esize * self.coff, self.lib_dtype, out.data_ptr(), B,
                                          self.C, S, self.cstride, _lib.stream_ptr())
        _lib.check(rc, "occd_cl_to_planar")
        return out[:, :, 0] if squeeze_d else out


def fold_bn(weight, bias, bn, eps=None):
    """conv -> BatchNorm(eval) == conv with w*scale and (b-mean)*scale+beta.  Returns fp32 (w, b)."""
    w = weight.detach().float()
    co = w.shape[0]
    b = bias.detach().float() if bias is not None else torch.zeros(co, device=w.device)
    if bn is None:
        return w, b
    e = bn.eps if eps is None else eps
    scale = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + e)
    shape = [co] + [1] * (w.dim() - 1)
    return w * scale.view(shape), (b - bn.running_mean.detach().float()) * scale + bn.bias.detach().float()


class ConvOp:
    """One planned implicit-GEMM launch (occd_conv_plan_create / occd_conv_run)."""

    def __init__(self, srcs, taps, tap_weights, bias, out_dims, out0=None, act="none", res1=None, res2=None,
                 stride=(1, 1, 1), omul=(1, 1, 1), oadd=(0, 0, 0), full_dims=None, out1=None, out1_mode="none",
                 out1_coff=0, impl=None, name="", res2_post=False, weight_buf=None, weight_per_image=False,
                 out0_exact=False, groups=None):
        """srcs: list[CL] (same B,D,H,W);  taps: [(src_idx, dz, dy, dx)];  tap_weights: list of fp32 [Cout, C_src]
        bias: fp32 [Cout];  out0/res1/res2: CL on the full output grid;  out1: CL (pre-activation bf16 copy) or
        fp32 planar tensor [B, C1, D, H, W] (mode "planar", written at channel out1_coff).
        groups: [(n_taps_of_group, (oadd_d, oadd_h, oadd_w))] -- several convolutions over the same sources in one
        launch, each with its own slice of `taps` and output offset (occd_conv_desc.n_groups; per-tap TC kernel)."""
        self.name = name
        dev = srcs[0].buf.device
        B, ID, IH, IW = srcs[0].dims
        for s in srcs:
            assert s.dims == (B, ID, IH, IW)
        Cout = int(bias.numel())
        Cout_pad = _round_up(Cout, 16)
        maxC = max(s.C for s in srcs)
        adt = srcs[0].buf.dtype
        for s in srcs:
            assert s.buf.dtype == adt
        esize = srcs[0].esize
        KC = chunk_channels(maxC, esize)
        Kpad = _round_up(maxC, KC)
        if weight_buf is not None:
            # weights produced at run time by another launch (CRP bmm): [n_taps, Cout_pad, Kpad] in the plan's dtype
            nset = B if weight_per_image else 1
            assert weight_buf.dtype == adt and tuple(weight_buf.shape) == (nset * len(taps), Cout_pad, Kpad)
            self.weight = weight_buf
        else:
            wp = torch.zeros(len(taps), Cout_pad, Kpad, dtype=torch.float32, device=dev)
            for i, (tp, w) in enumerate(zip(taps, tap_weights)):
                assert w.shape == (Cout, srcs[tp[0]].C), (w.shape, Cout, srcs[tp[0]].C)
                wp[i, :Cout, : w.shape[1]] = w
            self.weight = (round_tf32_(wp) if adt == torch.float32 else wp.to(torch.bfloat16)).contiguous()
        self.bias = torch.zeros(Cout_pad, dtype=torch.float32, device=dev)
        self.bias[:Cout] = bias.float()
        OD, OH, OW = out_dims
        fd = tuple(full_dims) if full_dims is not None else (OD, OH, OW)
        d = _lib.ConvDesc()
        if impl is None:
            impl = default_impl()
        if groups:
            impls = [_lib.CONV_IMPL_TC]
        elif impl is not None:
            impls = [impl]
        else:
            # auto: the candidates in order of preference, each tried until occd_conv_plan_create accepts one (its
            # geometry may still decline, e.g. when the weights and one stage do not fit in shared memory)
            impls = []
            if halox_eligible(srcs, taps, stride, omul, out_dims, Cout_pad, weight_buf):
                impls.append(_lib.CONV_IMPL_HALOX)
            if halo_eligible(srcs, taps, stride, omul, out_dims, Cout_pad, weight_buf):
                impls.append(_lib.CONV_IMPL_HALO)
            elif tcx_eligible(taps, stride, Cout_pad):
                impls.append(_lib.CONV_IMPL_TCX)
            impls.append(_lib.CONV_IMPL_TC)
        d.dtype = LIB_DTYPE[precision_of(adt)]
        d.n_src = len(srcs)
        for i, s in enumerate(srcs):
            assert s.d0 == srcs[0].d0 and s.buf.shape[1] == srcs[0].buf.shape[1]
            d.src[i] = s.full_ptr
            d.src_C[i], d.src_cstride[i], d.src_coff[i] = s.C, s.cstride, s.coff
        d.B, d.ID, d.IH, d.IW = B, srcs[0].buf.shape[1], IH, IW
        d.src_d0 = srcs[0].d0
        for i in range(3):
            d.stride[i], d.omul[i], d.oadd[i] = stride[i], omul[i], oadd[i]
        d.n_taps = len(taps)
        for i, (si, dz, dy, dx) in enumerate(taps):
            d.taps[i].src, d.taps[i].dz, d.taps[i].dy, d.taps[i].dx = si, dz, dy, dx
        if groups:
            assert sum(g[0] for g in groups) == len(taps) and len(groups) <= _lib.CONV_MAX_GROUPS
            d.n_groups, t0 = len(groups), 0
            for gi, (cnt, off) in enumerate(groups):
                d.group_tap0[gi] = t0
                t0 += cnt
                for i in range(3):
                    d.group_oadd[gi][i] = off[i]
            d.group_tap0[len(groups)] = t0
        d.weight, d.bias = self.weight.data_ptr(), self.bias.data_ptr()
        d.Cout, d.Cout_pad, d.Kpad = Cout, Cout_pad, Kpad
        d.weight_per_image = 1 if weight_per_image else 0
        d.OD, d.OH, d.OW = OD, OH, OW
        d.ODf, d.OHf, d.OWf = fd
        d.act = ACT[act]
        d.res2_post = 1 if res2_post else 0
        d.out0_exact = 1 if out0_exact else 0
        self._keep = [srcs, out0, res1, res2, out1]
        if out0 is not None:
            assert out0.dims == (B,) + fd and out0.C >= Cout and out0.buf.dtype == adt, (out0.dims, fd, out0.C, Cout)
            d.out0, d.out0_cstride, d.out0_coff = out0.ptr, out0.cstride, out0.coff
        for nm, r in (("res1", res1), ("res2", res2)):
            if r is not None:
                assert r.dims == (B,) + fd and r.C >= Cout and r.buf.dtype == adt
                setattr(d, nm, r.ptr)
                setattr(d, nm + "_cstride", r.cstride)
                setattr(d, nm + "_coff", r.coff)
        if out1_mode == "cl":
            assert out1.dims == (B,) + fd and out1.buf.dtype == adt
            d.out1_mode, d.out1 = _lib.OUT1_CL, out1.ptr
            d.out1_cstride, d.out1_coff = out1.cstride, out1.coff
        elif out1_mode == "planar":
            assert out1.dtype == torch.float32 and out1.is_contiguous() and tuple(out1.shape[2:]) == fd
            d.out1_mode, d.out1 = _lib.OUT1_F32_PLANAR, out1.data_ptr()
            d.out1_C, d.out1_coff = out1.shape[1], out1_coff
        self.desc = d
        self.flops = 2 * B * OD * OH * OW * Cout * sum(srcs[t[0]].C for t in taps)
        h = C.c_void_p()
        for impl in impls:
            d.impl = impl
            rc = _lib.lib().occd_conv_plan_create(C.byref(d), C.byref(h))
            if rc == 0:
                break
        _lib.check(rc, "occd_conv_plan_create(%s)" % name)
        self.handle = h
        self.impl = d.impl

    def info(self):
        arr = (C.c_int * 8)()
        _lib.check(_lib.lib().occd_conv_plan_info(self.handle, arr), "occd_conv_plan_info")
        return dict(zip(("TD", "TH", "TW", "N_tile", "KC", "stages", "grid_x", "grid_y"), list(arr)))

    def run(self, stream):
        _lib.check(_lib.lib().occd_conv_run(self.handle, stream), "occd_conv_run(%s)" % self.name)

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                _lib.lib().occd_conv_plan_destroy(self.handle)
        except Exception:
            pass


def conv_taps(weight, dilation=(1, 1, 1), padding=(0, 0, 0), src=0):
    """weight fp32 [Cout, Cin, kd, kh, kw] -> (taps, tap_weights) for a dense N-d convolution."""
    co, ci, kd, kh, kw = weight.shape
    taps, ws = [], []
    for a in range(kd):
        for b in range(kh):
            for c in range(kw):
                taps.append((src, a * dilation[0] - padding[0], b * dilation[1] - padding[1],
                             c * dilation[2] - padding[2]))
                ws.append(weight[:, :, a, b, c])
    return taps, ws


def _t3(v):
    return (v, v, v) if isinstance(v, int) else tuple(v)


def out_size(i, k, s, p, d):
    return (i + 2 * p - d * (k - 1) - 1) // s + 1


class Plan:
    """Ordered list of prepared launches (anything with .run(stream)) + named buffers."""

    def __init__(self, device, slab=None, precision=None):
        self.device = device
        self.precision = precision or default_precision()
        assert self.precision in PRECISIONS
        self.dtype = TORCH_DTYPE[self.precision]        # element type of every activation / GEMM weight buffer
        self.lib_dtype = LIB_DTYPE[self.precision]
        self.esize = 4 if self.precision == "tf32" else 2
        self.ops = []
        self.flops = 0
        self.graph, self.graph_ops = None, 0
        self.slab = slab            # parallel.SlabContext for the X-slab multi-GPU partition, else None
        self._exchanged = set()

    def alloc(self, B, D, H, W, C_):
        """3-D activations (D > 1) of a slab-partitioned plan get halo margins; everything else is dense."""
        halo = self.slab.halo if (self.slab is not None and D > 1) else 0
        return CL.alloc(B, D, H, W, C_, self.device, halo=halo, precision=self.precision)

    def kpad_for(self, C_):
        return _round_up(C_, chunk_channels(C_, self.esize))

    def pack_weights(self, w):
        """fp32 GEMM weights -> this plan's operand type (TF32-rounded fp32 or bf16)"""
        w = w.detach().float().contiguous()
        return round_tf32_(w.clone()) if self.precision == "tf32" else w.to(torch.bfloat16)

    def need_halo(self, src, taps, stride0, out_d):
        """Insert the neighbour exchange for `src` before a conv whose taps reach across the slab boundary."""
        if self.slab is None or src.halo == 0:
            return
        left = max(0, -min(t[1] for t in taps))
        right = max(0, (out_d - 1) * stride0 + max(t[1] for t in taps) - (src.dlen - 1))
        if left == 0 and right == 0:
            return
        if max(left, right) > src.halo or max(left, right) > src.dlen:
            raise RuntimeError("slab partition: a convolution reaches %d planes across the slab boundary but the slab "
                               "is %d planes thick (halo margin %d): use fewer ranks" % (max(left, right), src.dlen,
                                                                                       src.halo))
        key = src.buf.data_ptr()
        if key in self._exchanged:
            return
        self._exchanged.add(key)
        self.add(self.slab.exchange_op(src))

    def add(self, op):
        self.ops.append(op)
        self.flops += getattr(op, "flops", 0)
        return op

    # ---- dense convolution (2-D maps have D == 1) ----
    def conv(self, x, weight, bias, stride=1, padding=0, dilation=1, act="none", out=None, res1=None, res2=None,
             out1=None, out1_mode="none", out1_coff=0, name="conv", impl=None, res2_post=False, no_out0=False,
             out0_exact=False):
        """x: CL; weight fp32 [Cout,Cin,kd,kh,kw] (BN already folded); returns the output CL."""
        s, p, d = _t3(stride), _t3(padding), _t3(dilation)
        B, ID, IH, IW = x.dims
        co, ci, kd, kh, kw = weight.shape
        assert ci == x.C, (ci, x.C, name)
        od = (out_size(ID, kd, s[0], p[0], d[0]), out_size(IH, kh, s[1], p[1], d[1]),
              out_size(IW, kw, s[2], p[2], d[2]))
        if out is None and not no_out0:
            out = self.alloc(B, od[0], od[1], od[2], co)
        taps, ws = conv_taps(weight, d, p)
        self.need_halo(x, taps, s[0], od[0])
        self.add(ConvOp([x], taps, ws, bias, od, out0=out, act=act, res1=res1, res2=res2, stride=s, out1=out1,
                        out1_mode=out1_mode, out1_coff=out1_coff, name=name, impl=impl, res2_post=res2_post,
                        out0_exact=out0_exact))
        return out

    def conv_multi(self, srcs, weights, bias, paddings, dilations, act="none", out=None, res1=None, res2=None,
                   name="conv_multi", impl=None):
        """sum_i conv(srcs[i], weights[i]) with one accumulator (stride 1, 'same' geometry)."""
        B, ID, IH, IW = srcs[0].dims
        taps, ws = [], []
        for i, (w, p, d) in enumerate(zip(weights, paddings, dilations)):
            t, wl = conv_taps(w, _t3(d), _t3(p), src=i)
            taps += t
            ws += wl
        co = weights[0].shape[0]
        if out is None:
            out = self.alloc(B, ID, IH, IW, co)
        for i, src in enumerate(srcs):
            self.need_halo(src, [t for t in taps if t[0] == i], 1, ID)
        self.add(ConvOp(srcs, taps, ws, bias, (ID, IH, IW), out0=out, act=act, res1=res1, res2=res2, name=name,
                        impl=impl))
        return out

    def conv_transpose_k3s2(self, x, weight, bias, act="none", out=None, name="convT", impl=None, res_post=None):
        """ConvTranspose3d(kernel 3, stride 2, padding 1, output_padding 1) as 8 sub-pixel phase convolutions.
        weight fp32 [Cin, Cout, 3, 3, 3] (torch layout, BN folded over Cout).  out[o] += x[i] w[k], o = 2i-1+k:
        even o=2j uses (k=1,i=j); odd o=2j+1 uses (k=2,i=j) and (k=0,i=j+1)."""
        B, ID, IH, IW = x.dims
        ci, co = weight.shape[:2]
        assert ci == x.C
        if out is None:
            out = self.alloc(B, 2 * ID, 2 * IH, 2 * IW, co)
        sel = {0: [(1, 0)], 1: [(2, 0), (0, 1)]}  # parity -> [(kernel index, input offset)]
        self.need_halo(x, [(0, 1, 0, 0)], 1, ID)
        phases = []
        for pd in (0, 1):
            for ph in (0, 1):
                for pw in (0, 1):
                    taps, ws = [], []
                    for (ka, oa) in sel[pd]:
                        for (kb, ob) in sel[ph]:
                            for (kc, oc) in sel[pw]:
                                taps.append((0, oa, ob, oc))
                                ws.append(weight[:, :, ka, kb, kc].t())
                    phases.append(((pd, ph, pw), taps, ws))
        if impl is None:
            impl = default_impl()
        grouped = impl in (None, _lib.CONV_IMPL_TC) and os.environ.get("OCCDEPTH_CONVT_GROUPED", "1") == "1"
        if grouped:
            # ONE launch: the 8 phases as tap groups of the per-tap kernel, largest group first (the persistent grid
            # walks the tiles group-major, so every CTA gets the same share of each phase)
            phases.sort(key=lambda p: -len(p[1]))
            self.add(ConvOp([x], [t for p in phases for t in p[1]], [w for p in phases for w in p[2]], bias,
                            (ID, IH, IW), out0=out, act=act, omul=(2, 2, 2), res2=res_post, res2_post=True,
                            full_dims=(2 * ID, 2 * IH, 2 * IW), name=name,
                            groups=[(len(p[1]), p[0]) for p in phases]))
            return out
        for (pd, ph, pw), taps, ws in phases:
            self.add(ConvOp([x], taps, ws, bias, (ID, IH, IW), out0=out, act=act, omul=(2, 2, 2),
                            res2=res_post, res2_post=True,
                            oadd=(pd, ph, pw), full_dims=(2 * ID, 2 * IH, 2 * IW),
                            name="%s.p%d%d%d" % (name, pd, ph, pw), impl=impl))
        return out

    def run(self, stream=None):
        """Replays the launches on the current stream (through a captured CUDA graph when enabled)."""
        if stream is None and self.graph is not None:
            self.graph.replay()
            st = _lib.stream_ptr()
            for op in self.ops[self.graph_ops:]:
                op.run(st)
            return
        st = _lib.stream_ptr() if stream is None else stream
        for op in self.ops:
            op.run(st)

    def capture(self):
        """Capture the launch sequence into a CUDA graph (buffers are static, so replay is valid).  Communication
        ops (NCCL halo exchange / all-gather of the slab partition) are not captured: the graph covers the ops
        before the first of them (the replicated 2D network and the lift), the rest is launched eagerly."""
        self.graph = None
        n = len(self.ops)
        for i, op in enumerate(self.ops):
            if getattr(op, "name", "") in ("halo_exchange", "all_gather"):
                n = i
                break
        self.run()                      # warm-up outside capture (lazy module loading, func attributes)
        torch.cuda.synchronize()
        if n == 0:
            return None
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            st = _lib.stream_ptr()
            for op in self.ops[:n]:
                op.run(st)
        self.graph, self.graph_ops = g, n
        return g

    def profile(self):
        """Per-launch device times (CUDA events on the launching stream); returns [(name, ms, flops)]."""
        st = _lib.stream_ptr()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(self.ops) + 1)]
        # park the GPU on a spin kernel while the host enqueues everything: the event deltas then measure
        # back-to-back device execution instead of host launch latency
        torch.cuda._sleep(int(1.9e9 * 0.04))
        evs[0].record()
        for i, op in enumerate(self.ops):
            op.run(st)
            evs[i + 1].record()
        torch.cuda.synchronize()
        return [(getattr(op, "name", "?"), evs[i].elapsed_time(evs[i + 1]), getattr(op, "flops", 0))
                for i, op in enumerate(self.ops)]


class FnOp:
    """A prepared non-conv launch: fn(stream) -> rc."""

    def __init__(self, fn, name, keep=()):
        self.fn, self.name, self._keep = fn, name, keep

    def run(self, stream):
        _lib.check(self.fn(stream), self.name)


def kpad_for(C_, esize=2):
    return _round_up(C_, chunk_channels(C_, esize))
