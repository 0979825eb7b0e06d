"""Per-role clock64 timeline of CTA 0 of the persistent conv kernel: python tools/conv_trace.py <shape>"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402

dev = torch.device("cuda")
buf = torch.zeros(64 * 8, dtype=torch.int64, device=dev)
import conv_bench  # noqa: E402
from occdepth_b200 import _lib  # noqa: E402
from occdepth_b200.engine import CL, Plan  # noqa: E402

_lib.check(_lib.lib().occd_conv_debug_trace(buf.data_ptr()), "occd_conv_debug_trace")
PREC = os.environ.get("OCCDEPTH_PRECISION", "tf32")

n = sys.argv[1]
dims, ci, co, k, dl, act = conv_bench.SHAPES[n]
plan = Plan(dev, precision=PREC)
x = plan.alloc(1, dims[0], dims[1], dims[2], ci)
x.buf.normal_()
w = torch.randn(co, ci, *k, device=dev) / (ci * k[0] * k[1] * k[2]) ** 0.5
plan.conv(x, w, torch.randn(co, device=dev), padding=tuple(dl * (kk - 1) // 2 for kk in k), dilation=dl, act=act)
for _ in range(3):
    plan.run()
torch.cuda.synchronize()
t = buf.cpu().view(64, 8)
t0 = int(t[0, 0])
print(n, plan.ops[0].info())
print("tile: prod_start prod_end | mma_start mma_end | epi_wait epi_go epi_end   (cycles since first stamp)")
for j in range(12):
    print(j, [int(v) - t0 if v else None for v in t[j, :7]])
