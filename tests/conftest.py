import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu on the GPU box")


def pytest_collection_modifyitems(config, items):
    # kernel-level GPU tests first: a broken kernel fails in seconds, before the full-size model tests spend minutes
    # on CPU oracle forwards -- and the process's first launches are the library's own tcgen05 kernels
    order = ["test_gpu_conv", "test_gpu_ops", "test_gpu_sfa", "test_gpu_unet3d", "test_gpu_net2d", "test_gpu_golden",
             "test_gpu_slab", "test_gpu_dropin", "test_gpu_zz_widening", "test_gpu_config4", "test_gpu_config2"]

    def key(item):
        mod = item.module.__name__.rsplit(".", 1)[-1]
        return order.index(mod) if mod in order else -1
    items.sort(key=key)        # stable: non-GPU modules keep their order in front
