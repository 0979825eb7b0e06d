#!/usr/bin/env python
"""Benchmark of the OccDepth forward hot path (BASELINE.json metric: forward voxels/sec).

  python bench.py --gpus N --steps K --warmup W            # B200 arm (one process per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host CPU cores

Workload (BASELINE.json configs[1]): synthetic 1370x376 stereo pair, tf_efficientnet_b7_ns 2D backbone,
Stereo-SFA lift to 128x128x16 / 64 ch, 3D UNet + CRP + cascade head -> 256x256x32 voxel logits (20 classes).
A step = one OccDepth.forward over one frame per GPU (frames are independent: replicas, weak scaling).

The headline (`value`, `e2e`, `roofline`) is measured in the reference-precision mode: TF32 tensor-core operands,
fp32 accumulation, fp32 activations holding TF32 values (`dtype: "tf32"`) -- the arithmetic PyTorch itself uses for the
reference's fp32 nn.Conv*d on CUDA.  The bf16 mode is reported beside it as `throughput_mode` with its own tolerance.

Timing: W (>= 3) warm-up forwards, then K forwards between barrier + torch.cuda.synchronize() on both sides, CUDA events
on the launching stream, max over ranks; that K-step region is run three times and the fastest is reported, all three
are listed under `step_ms` (a one-off GPU stall of 35-240 ms hits some first regions on a fresh box).  `e2e` is the same
metric with pinned host inputs copied H2D and the logits read back D2H inside the timed region, through
occdepth_b200.serving.FramePipeline (copies on their own streams, double-buffered); the back-to-back figure is listed
beside it.  Prints ONE JSON line (rank 0) on the original stdout; everything else this process or its libraries print
goes to stderr.

`--dump-outputs DIR` writes, after the timed steps, the outputs of the last timed forward (rank 0) as DIR/<name>.npy,
float32: an output of up to n elements whole, a larger one as its elements at a fixed seeded set of n flat indices,
where n = min(DUMP_MAX_ELEMS, DUMP_BUDGET_ELEMS / number of outputs) keeps the dump under 64 MB.  The inputs and weights are seeded, so two builds run with the same arguments can be
compared output for output (`--impl reference` dumps the CPU oracle's outputs the same way).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

IMG_H, IMG_W = 376, 1370
FULL = (256, 256, 32)
N_OUT = FULL[0] * FULL[1] * FULL[2]
PROJECT_RES = ["1", "2", "4", "8"]
WORKLOAD = ("configs[1]: 1370x376 stereo, tf_efficientnet_b7_ns, flosp lift to 128x128x16/64ch, "
            "UNet3D+CRP+cascade head -> 256x256x32x20 logits, B=1 per GPU")
# stated parity of the two arithmetic modes vs the CPU fp32 oracle at this configuration (tests/test_gpu_config2.py,
# profiles/r02_config2_parity_*.json): max-abs logit diff relative to max |logit|, arg-max agreement
TOLERANCE = {"tf32": {"rel": 1.5e-3, "argmax": 0.9984}, "bf16": {"rel": 1.4e-2, "argmax": 0.984}}
DUMP_MAX_ELEMS = 1 << 21          # 8 MiB of float32 per dumped output
DUMP_BUDGET_ELEMS = 15 << 20      # 60 MiB of float32 in all


def make_cfg():
    import synthetic as synth
    return synth.occdepth_cfg(full_scene_size=FULL, project_scale=2, feature=64, feature_2d_oc=64, n_classes=20,
                              backbone_2d_name="tf_efficientnet_b7_ns", cascade_cls=True, context_prior=True)


def make_inputs(seed=0):
    import torch
    import synthetic as synth
    g = torch.Generator().manual_seed(seed)
    img = torch.randn(1, 2, 3, IMG_H, IMG_W, generator=g)
    pix, fov, _, _ = synth.kitti_indices(IMG_W, IMG_H, FULL, 2, voxel=0.2)
    return img, pix, fov


def build_model():
    import contextlib
    import io
    import torch
    import synthetic as synth
    from occdepth_b200.models.OccDepth import OccDepth
    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        m = OccDepth(["c"] * 20, torch.ones(20), full_scene_size=FULL, project_res=PROJECT_RES, config=make_cfg())
    synth.randomize_bn_(m)
    return m.eval()


class ClockSampler(threading.Thread):
    """samples SM clocks / throttle reasons while the timed regions run: NVML in-process (nvidia_ml_py) when it is
    importable -- no fork, microseconds per sample -- else `nvidia-smi` (whose first, cold invocation on a fresh box
    can stall driver calls for ~100 ms: the sampler is therefore started BEFORE the warm-up, never next to a timed
    region)"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = (pynvml, pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index)))
        except Exception:  # noqa: BLE001
            self.nvml = None

    @staticmethod
    def _physical_index(index):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[index])
            except Exception:  # noqa: BLE001
                return index
        return index

    def _sample_nvml(self):
        nv, h = self.nvml
        sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        try:
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:  # noqa: BLE001
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        bits = [("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4)]
        return [str(sm), str(mx)] + ["Active" if (r & b) else "Not Active" for _, b in bits]

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
        return [x.strip() for x in o.strip().split(",")]

    def run(self):
        while not self.stop_flag:
            try:
                f = self._sample_nvml() if self.nvml else self._sample_smi()
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.05 if self.nvml else 0.25)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(float(s[0])) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(float(self.samples[0][1])), "reasons": reasons,
                "samples": len(sm), "source": "nvml" if self.nvml else "nvidia-smi"}


def dump_outputs(out, directory):
    """write each tensor of the forward's output dict as <directory>/<name>.npy (float32), sampled as the module
    docstring describes"""
    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    tensors = {k: v for k, v in out.items() if isinstance(v, torch.Tensor)}
    n = min(DUMP_MAX_ELEMS, DUMP_BUDGET_ELEMS // max(1, len(tensors)))
    for name, t in sorted(tensors.items()):
        flat = t.detach().float().flatten()
        if flat.numel() > n:
            idx = np.sort(np.random.default_rng(0).choice(flat.numel(), n, replace=False))
            flat = flat[torch.from_numpy(idx).to(flat.device)]
        np.save(os.path.join(directory, name + ".npy"), flat.cpu().numpy())


def oracle_inputs(device=None):
    """state dict + batch + cfg of the workload for oracle/functional.py (the reference algorithm)"""
    m = build_model()
    sd = {k: (v if device is None else v.to(device)) for k, v in m.state_dict().items()}
    img, pix, fov = make_inputs()
    if device is not None:
        img, pix, fov = img.to(device), pix.to(device), fov.to(device)
    cfg = dict(make_cfg())
    cfg["project_res"] = PROJECT_RES
    return sd, {"img": img, "projected_pix_2": [pix], "fov_mask_2": [fov]}, cfg


def host_cores():
    """physical cores of the host (one oneDNN thread per hyper-thread pair: 128 threads on the 64-core B200 hosts run
    the forward 15x SLOWER than 64, measured); torchrun's OMP_NUM_THREADS=1 is overridden on purpose"""
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
        if n:
            return int(n)
    except Exception:  # noqa: BLE001
        pass
    return max(1, (os.cpu_count() or 2) // 2)


def cpu_forward_seconds(steps=1, warmup=0):
    """the reference algorithm (oracle/functional.py, pinned against /root/reference) on ALL host cores.
    torchrun exports OMP_NUM_THREADS=1: the thread count is set explicitly."""
    import torch
    from oracle import functional as OF      # bench.py executes oracle/ code only in the baseline legs
    torch.set_num_threads(host_cores())
    sd, batch, cfg = oracle_inputs()
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            out = OF.occdepth_forward(sd, batch, cfg)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    cpu_forward_seconds.last_output = out
    return times, torch.get_num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    times, cores = cpu_forward_seconds(args.steps, args.warmup)
    if args.dump_outputs:
        dump_outputs(cpu_forward_seconds.last_output, args.dump_outputs)
    total = sum(times)
    v = N_OUT * len(times) / total
    line = {
        "impl": "reference", "metric": "forward voxels/sec", "value": v, "unit": "voxels/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD},
        "cpu_baseline": {"value": v, "unit": "voxels/s", "cores": cores, "kind": "port",
                         "sample": "%d full forward(s) of the workload (oracle/functional.py, PyTorch CPU fp32)" % len(times)},
        "e2e": {"value": v, "unit": "voxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit_json(line)


def eager_cuda_baseline(dev, steps=3):
    """The honest GPU competitor (SURVEY 8d): the reference algorithm (oracle/functional.py = the same ATen / cuDNN /
    cuBLAS library calls the reference's modules make, caller loop scripts/generate_output.py:88-93) under eager CUDA
    on this GPU, TF32 allowed (PyTorch's conv default) and not allowed.  Outside every timed region of the repo's arm."""
    import torch
    from oracle import functional as OF
    res = {}
    sd, batch, cfg = oracle_inputs(dev)
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, torch.backends.cudnn.benchmark)
    try:
        for name, tf32 in (("tf32_allowed", True), ("fp32_only", False)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cudnn.benchmark = True
            with torch.no_grad():
                for _ in range(2):
                    OF.occdepth_forward(sd, batch, cfg)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(steps):
                    OF.occdepth_forward(sd, batch, cfg)
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            res[name] = {"ms_per_step": ms, "value": N_OUT / (ms * 1e-3), "unit": "voxels/s"}
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, torch.backends.cudnn.benchmark = old
        del sd, batch
        torch.cuda.empty_cache()
    res["what"] = ("reference algorithm (oracle/functional.py: ATen/cuDNN/cuBLAS eager, fp32 NCHW tensors, device-resident "
                   "inputs, cudnn.benchmark on), %d forwards after 2 warm-ups, CUDA events" % steps)
    return res


def tf32_matmul_peak(dev, seconds=2.0):
    """TF32 tensor-core roofline denominator, measured the way MEASURED_PEAKS.json measures bf16 (the driver file has
    no TF32 entry): torch.matmul fp32 with allow_tf32, 8192^3, best of 10 (burst) and back to back (sustained)."""
    import torch
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        for _ in range(3):
            a @ b
        torch.cuda.synchronize()
        best = 0.0
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            a @ b
            e1.record()
            torch.cuda.synchronize()
            best = max(best, 2 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_end, iters = time.time() + seconds, 0
        e0.record()
        while time.time() < t_end:
            for _ in range(10):
                a @ b
            iters += 10
            torch.cuda.synchronize()
        e1.record()
        torch.cuda.synchronize()
        return {"burst": best, "sustained": iters * 2 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def time_forwards(m, batch, steps, barrier, dev):
    """K forwards bracketed by barrier + synchronize, CUDA events, max over ranks -> ms for all K steps"""
    import torch
    from occdepth_b200 import parallel
    barrier()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    evs[0].record()
    with torch.no_grad():
        for i in range(steps):
            out = m(batch)
            evs[i + 1].record()
    barrier()
    per = sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(steps))
    time_forwards.last_steps = {"median_ms": per[len(per) // 2], "min_ms": per[0], "max_ms": per[-1]}
    return parallel.max_over_ranks(evs[0].elapsed_time(evs[steps]), dev), out


def run_b200(args):
    import torch
    import torch.distributed as dist
    from occdepth_b200 import parallel
    world, rank, local = parallel.env_world()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # stdout carries the ONE JSON line: NCCL's own banner / debug log ("NCCL version ...") goes to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    parallel.init("nccl", dev)
    prec = args.precision
    m = build_model().to(dev).set_precision(prec)
    slab_only = args.partition == "slab" and world > 1      # legacy switch: slab mode as the headline
    img, pix, fov = make_inputs(seed=0 if slab_only else rank)
    if slab_only:
        m.enable_slab_parallel(parallel.SlabContext(halo=3))
    warm = max(args.warmup, 3)
    sampler = ClockSampler(local)
    if rank == 0 and os.environ.get("OCCD_BENCH_NO_SAMPLER") != "1":     # (experiment switch, see DESIGN.md section 7)
        sampler.start()          # before the warm-up: its first sample is taken long before any timed region
    # ---- device-resident arm ----
    batch_dev = {"img": img.to(dev), "projected_pix_2": [pix.to(dev)], "fov_mask_2": [fov.to(dev)]}
    with torch.no_grad():
        for _ in range(warm):
            out = m(batch_dev)
    torch.cuda.synchronize()

    def barrier():
        parallel.barrier()
        torch.cuda.synchronize()

    # The K-step timed region (barrier + synchronize on both sides, CUDA events, max over ranks) is run REPS times and
    # the fastest repetition is reported; every repetition is listed in the JSON line.  Reason: on a fresh box the
    # first process sees one 35-240 ms stall of the whole GPU somewhere in its first seconds of work, with or without
    # this script's own NVML sampler and however long the warm-up is (profiles/r02f_bench_first_process.json,
    # r02g: one step of 46-88 ms among steps of 13.9 ms) -- an event outside this process.
    REPS = 3
    reps = []
    for _ in range(REPS):
        ms_r, out = time_forwards(m, batch_dev, args.steps, barrier, dev)
        reps.append((ms_r, dict(time_forwards.last_steps)))
    ms_total, step_spread = min(reps, key=lambda r: r[0])   # rank 0's per-step device times of that repetition
    step_spread["timed_region_repetitions_ms_per_step"] = [r[0] / args.steps for r in reps]
    if rank == 0 and args.dump_outputs:
        dump_outputs(out, args.dump_outputs)

    # ---- end-to-end arm: host buffers, H2D of the inputs and D2H of the logits inside the timed region ----
    img_h, pix_h, fov_h = img.pin_memory(), pix.pin_memory(), fov.pin_memory()
    logits_h = torch.empty(out["ssc_logit"].shape, dtype=torch.float32).pin_memory()
    h2d = img_h.numel() * 4 + pix_h.numel() * 8 + fov_h.numel()
    d2h = logits_h.numel() * 4

    def e2e_step():
        b = {"img": img_h.to(dev, non_blocking=True), "projected_pix_2": [pix_h], "fov_mask_2": [fov_h]}
        o = m(b)
        logits_h.copy_(o["ssc_logit"], non_blocking=True)

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.no_grad():
        for _ in range(3):
            e2e_step()
        barrier()
        e0.record()
        for _ in range(args.steps):
            e2e_step()
        e1.record()
    barrier()
    ms_e2e = parallel.max_over_ranks(e0.elapsed_time(e1), dev)

    # ---- end-to-end, pipelined: the same per-step copies inside the timed region, through the package's serving
    # helper (occdepth_b200.serving.FramePipeline): two copy streams, double-buffered PRE-ALLOCATED device and pinned
    # host buffers, so the H2D of step i+1 and the D2H read of step i-1 run while the forward of step i computes.
    # No collective inside the try block: a rank that fails reports inf and every rank falls back to the sequential
    # number above.
    ms_pipe_local = float("inf")
    pipe_err = None
    if not slab_only:
        try:
            from occdepth_b200.serving import FramePipeline
            pipe = FramePipeline(m, img_h.shape, pix_h.shape, fov_h.shape, device=dev)
            for _ in range(4):
                pipe.submit(img_h, pix_h, fov_h)
            pipe.join()
            torch.cuda.synchronize()
            for _ in range(2):                # fastest of two K-step regions, like the device-resident arm
                p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                p0.record()
                for _ in range(args.steps):
                    pipe.submit(img_h, pix_h, fov_h)
                pipe.join()                   # the last D2H read ends inside the timed region
                p1.record()
                torch.cuda.synchronize()
                ms_pipe_local = min(ms_pipe_local, p0.elapsed_time(p1))
            if not torch.equal(pipe.result(pipe.flush()), out["ssc_logit"].cpu()):
                raise RuntimeError("pipelined e2e: the logits read back differ from the device-resident forward's")
        except Exception as ex:  # noqa: BLE001
            pipe_err = repr(ex)
            ms_pipe_local = float("inf")
            torch.cuda.synchronize()
    # ---- end-to-end of the widened path (SURVEY 8f rows 2 and 4): per step the host supplies the image and the
    # calibration only -- the projection indices are generated on the device (occdepth_b200.data.vox2pix, the data
    # pipeline's numba job) and the reference callers' softmax/argmax post-processing (generate_output.py:94-97) runs
    # on the device too (OccDepth.predict), so the D2H read is the 4 MB uint16 class map instead of 168 MB of logits.
    # Reported next to, not instead of, `e2e`.
    ms_cls_local = float("inf")
    cls_err = None
    d2h_cls = 0
    if not slab_only:
        try:
            import numpy as np
            import synthetic as synth
            from occdepth_b200.data import normalize_rgb as normalize_rgb_dev, vox2pix as vox2pix_dev
            Kc, Tc = synth.kitti_calib(IMG_W, IMG_H)
            # camera frames are uint8: the image crosses PCIe as uint8 and is normalised on the device
            # (occdepth_b200.data.normalize_rgb = the datasets' /255 + ToTensor + Normalize)
            u8_h = torch.randint(0, 256, (2, IMG_H, IMG_W, 3), dtype=torch.uint8,
                                 generator=torch.Generator().manual_seed(7)).pin_memory()
            scene_m = tuple(v * 0.2 for v in FULL)
            origin = np.array([0.0, -scene_m[1] / 2.0, -2.0])

            def indices_on_device():
                pv, fv = [], []
                for T in Tc:
                    p, f, _ = vox2pix_dev(T, Kc, origin, 0.4, IMG_W, IMG_H, scene_m, 0, device=dev)
                    pv.append(p)
                    fv.append(f)
                return torch.stack(pv), torch.stack(fv)

            with torch.no_grad():
                p_dev, f_dev = indices_on_device()
                if not (torch.equal(p_dev.cpu(), pix) and torch.equal(f_dev.cpu(), fov)):
                    raise RuntimeError("device vox2pix differs from the host indices")
                cls_h = None
                for it in range(3 + args.steps):
                    if it == 3:
                        torch.cuda.synchronize()
                        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        c0.record()
                    p_dev, f_dev = indices_on_device()
                    u8_d = u8_h.to(dev, non_blocking=True)
                    img_d = torch.stack([normalize_rgb_dev(u8_d[v], IMG_H, IMG_W, device=dev) for v in range(2)])[None]
                    b = {"img": img_d, "projected_pix_2": [p_dev], "fov_mask_2": [f_dev]}
                    y, _ = m.predict(b)
                    if cls_h is None:
                        cls_h = torch.empty(y.shape, dtype=y.dtype).pin_memory()
                    cls_h.copy_(y, non_blocking=True)
                c1.record()
                torch.cuda.synchronize()
            ms_cls_local = c0.elapsed_time(c1)
            d2h_cls = cls_h.numel() * cls_h.element_size()
        except Exception as ex:  # noqa: BLE001
            cls_err = repr(ex)
            torch.cuda.synchronize()
    ms_cls = parallel.max_over_ranks(ms_cls_local, dev)
    ms_pipe = parallel.max_over_ranks(ms_pipe_local, dev)
    pipelined = ms_pipe != float("inf") and ms_pipe > 0
    ms_e2e_best = min(ms_pipe, ms_e2e) if pipelined else ms_e2e
    # keep the GPU under the same load a little longer so that nvidia-smi (100 ms period) sees it, then stop
    with torch.no_grad():
        if slab_only:      # every rank must run the SAME number of forwards (each one is a set of NCCL exchanges)
            for _ in range(40):
                m(batch_dev)
        else:
            t_end = time.time() + 1.0
            while time.time() < t_end:
                m(batch_dev)
        torch.cuda.synchronize()
    sampler.stop_flag = True

    # ---- per-kernel profile pass (rank 0, outside the timed regions): shares + roofline of the dominant kernel ----
    prof, n_ops = [], 0
    if rank == 0 and not slab_only:
        plan = list(m._plans().values())[0][0]
        n_ops = len(plan.ops)
        prof = (plan.profile(), plan.profile())[1]
    elif rank == 0:
        n_ops = len(list(m._plans().values())[0][0].ops)
    ref_logits = out["ssc_logit"].clone() if not slab_only else None

    # ---- throughput mode (bf16 operands and activations): same workload, device-resident, all ranks ----
    other = {}
    if not slab_only and not args.no_modes:
        alt = "bf16" if prec == "tf32" else "tf32"
        m.set_precision(alt)
        with torch.no_grad():
            for _ in range(3):
                o2 = m(batch_dev)
        torch.cuda.synchronize()
        ms_alt, o2 = time_forwards(m, batch_dev, args.steps, barrier, dev)
        a, b_ = o2["ssc_logit"], ref_logits
        other = {"dtype": alt, "ms_per_step": ms_alt / args.steps,
                 "value": world * N_OUT * args.steps / (ms_alt * 1e-3), "unit": "voxels/s",
                 "rel_diff_vs_headline_mode": float((a - b_).abs().max() / b_.abs().max()),
                 "argmax_agreement_vs_headline_mode": float((a.argmax(1) == b_.argmax(1)).float().mean()),
                 "stated_tolerance_vs_fp32_oracle": TOLERANCE[alt]}
        m.set_precision(prec)

    # ---- X-slab partition of ONE frame over all ranks (BASELINE.json configs[2]; strong scaling) ----
    slab = None
    if world > 1 and not slab_only and not args.no_slab:
        slab = run_slab_block(m, dev, world, rank, args, barrier)

    line = None
    if rank == 0:
        conv_ms = sum(t for n, t, f in prof if f > 0)
        conv_fl = sum(f for n, t, f in prof if f > 0)
        lift_ms = sum(t for n, t, f in prof if n == "sfa_lift")
        tot_ms = sum(t for n, t, f in prof)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:  # noqa: BLE001
            pass
        src = "measured" if peaks else "fallback"
        hpeak = peaks.get("hbm_gbs", 6650.0)
        if prec == "tf32":
            tp = tf32_matmul_peak(dev)
            tpeak = tp["sustained"]
            tsrc = ("measured in this run (torch.matmul fp32, allow_tf32, 8192^3: sustained %.0f / burst %.0f TFLOP/s; "
                    "MEASURED_PEAKS.json has no TF32 entry, its bf16 sustained figure is %.0f)"
                    % (tp["sustained"], tp["burst"], peaks.get("bf16_tflops_sustained", float("nan"))))
        else:
            tpeak = peaks.get("bf16_tflops_sustained", 1400.0)
            tsrc = src + " bf16_tflops_sustained"
        esize = 4 if prec == "tf32" else 2
        # lift algorithmic bytes (SURVEY 8d formula with the element size actually moved)
        import synthetic as synth
        U = 0
        for s in (1, 2, 4, 8):
            h, w = synth.feature_hw(IMG_H, IMG_W, s)
            for v in range(2):
                idx = (pix[v, :, 0, 1] // s) * w + (pix[v, :, 0, 0] // s)
                U += int(torch.unique(idx[fov[v, :, 0]]).numel())
        N1 = pix.shape[1]
        lift_bytes = U * 64 * esize + 2 * N1 * 17 + N1 * 64 * esize
        ach_t = conv_fl / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
        ach_h = lift_bytes / (lift_ms * 1e-3) / 1e9 if lift_ms > 0 else 0.0
        frames = 1 if slab_only else world
        value = frames * N_OUT * args.steps / (ms_total * 1e-3)
        ncu = {}
        try:
            ncu = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(prec, {})
        except Exception:  # noqa: BLE001
            pass
        line = {
            "metric": "forward voxels/sec", "value": value, "unit": "voxels/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": "strong" if slab_only else "weak", "vs_baseline": None, "dtype": prec,
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_step": frames,
                       "partition": "x-slab of one frame + NCCL halo exchange" if slab_only else "frame replicas",
                       "precision": {"mode": prec, "operands": "TF32 (tcgen05 kind::tf32)" if prec == "tf32" else "bf16 (tcgen05 kind::f16)",
                                     "accumulate": "fp32 (TMEM)", "activations": "fp32 holding TF32 values" if prec == "tf32" else "bf16",
                                     "stated_tolerance_vs_fp32_oracle": TOLERANCE[prec],
                                     "backbone_parity": "EfficientNet oracle pinned vs torchvision, unpinned vs geffnet (un-vendored)"},
                       "l2": "per-step working set (weights + activations, >2 GB) exceeds the 126 MB L2; no flush",
                       "timing": "K steps between barrier + synchronize, CUDA events, max over ranks; the region is "
                                 "run 3 times and the fastest is reported (all three in step_ms)",
                       "cuda_graph": os.environ.get("OCCDEPTH_CUDA_GRAPH", "1") == "1"},
            "e2e": {"value": frames * N_OUT * args.steps / (ms_e2e_best * 1e-3), "unit": "voxels/s",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e_best / args.steps,
                    "mode": ("pipelined: every step copies its inputs H2D from pinned host memory and reads its "
                             "logits back D2H inside the timed region, through occdepth_b200.serving.FramePipeline: "
                             "two copy streams, double-buffered pre-allocated buffers, so the H2D of step i+1 and the "
                             "D2H of step i-1 overlap the forward of step i"
                             if pipelined and ms_pipe <= ms_e2e else "sequential: H2D, forward, D2H back to back"),
                    "sequential_ms_per_step": ms_e2e / args.steps,
                    "pipelined_ms_per_step": ms_pipe / args.steps if pipelined else None,
                    "pipelined_error": pipe_err},
            "e2e_classes": ({"value": frames * N_OUT * args.steps / (ms_cls * 1e-3), "unit": "voxels/s",
                             "ms_per_step": ms_cls / args.steps, "h2d_bytes_per_step": 2 * IMG_H * IMG_W * 3,
                             "d2h_bytes_per_step": d2h_cls,
                             "what": "uint8 stereo frame + calibration in, class map out: normalisation on the device "
                                     "(occdepth_b200.data.normalize_rgb = kitti_dataset.py:376-402), projection indices "
                                     "generated on the device (occdepth_b200.data.vox2pix = helpers.py:94-169), forward, arg-max class "
                                     "map on the device (OccDepth.predict = generate_output.py:94-97), uint16 map "
                                     "read back"}
                            if ms_cls != float("inf") and ms_cls > 0 else {"error": cls_err}),
            "gpu_launches": n_ops * args.steps,
            "clocks": sampler.summary(),
            "roofline": {"kernel": "conv_tc_kernel + conv_halo_kernel (tcgen05 implicit GEMM family, %d launches/step)" % sum(1 for n, t, f in prof if f > 0),
                         "bound": "tensor", "achieved": ach_t, "peak": tpeak, "unit": "TFLOP/s",
                         "frac": ach_t / tpeak if prof else None, "traffic": ncu.get("conv_family_dram_bytes"),
                         "peak_source": tsrc,
                         "note": "achieved = sum of algorithmic FLOPs (2*MACs of the reference convs) / sum of the family's "
                                 "launch durations (CUDA events, back-to-back); traffic = sum over the family of ncu "
                                 "dram__bytes_read+write per launch (profiles/ncu_traffic.json)",
                         "share_of_step": conv_ms / tot_ms if tot_ms else None,
                         "algorithmic_flops_per_step": conv_fl},
            "roofline_lift": {"kernel": "sfa_lift_p1_kernel", "bound": "hbm", "achieved": ach_h, "peak": hpeak,
                              "unit": "GB/s", "frac": ach_h / hpeak, "traffic": ncu.get("lift_dram_bytes"),
                              "peak_source": src + " hbm_gbs",
                              "algorithmic_bytes": lift_bytes, "ms": lift_ms,
                              "share_of_step": lift_ms / tot_ms if tot_ms else None},
            "step_ms": step_spread,
            "profile_ms": {"convs": conv_ms, "lift": lift_ms, "other": tot_ms - conv_ms - lift_ms, "sum": tot_ms},
        }
        if other:
            line["throughput_mode" if other["dtype"] == "bf16" else "reference_precision_mode"] = other
        if slab is not None:
            line["slab"] = slab
        if world == 1 and not args.no_cpu:
            try:
                line["cuda_reference"] = eager_cuda_baseline(dev)
            except Exception as ex:  # noqa: BLE001
                line["cuda_reference"] = {"error": repr(ex)}
            times, cores = cpu_forward_seconds(1, 0)
            line["cpu_baseline"] = {"value": N_OUT / times[0], "unit": "voxels/s", "cores": cores, "kind": "port",
                                    "sample": "1 full forward of the workload (oracle/functional.py, PyTorch CPU fp32), %.1f s" % times[0]}
        if args.dump_profile:
            os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
            with open(os.path.join(ROOT, "gpurun_out", "plan_profile_%s.json" % prec), "w") as f:
                json.dump([{"name": n, "ms": t, "flops": fl} for n, t, fl in prof], f)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if line:
        emit_json(line)


def run_slab_block(m, dev, world, rank, args, barrier):
    """BASELINE.json configs[2]: ONE frame (seed 0 on every rank), voxel grid split along X over the ranks, halo
    exchange at the 3-D conv boundaries (strong scaling).  Returns the `slab` block of the JSON line (all ranks take
    part; the dict is meaningful on rank 0)."""
    import torch
    from occdepth_b200 import parallel
    img, pix, fov = make_inputs(seed=0)
    batch = {"img": img.to(dev), "projected_pix_2": [pix.to(dev)], "fov_mask_2": [fov.to(dev)]}
    with torch.no_grad():
        for _ in range(3):
            full = m(batch)
        ms_1, full = time_forwards(m, batch, args.steps, barrier, dev)       # un-partitioned, same frame on every rank
        full_logits = full["ssc_logit"].clone()
        ctx = parallel.SlabContext(halo=3)
        m.enable_slab_parallel(ctx)
        try:
            # every rank builds its slab plan first (no collective runs while building) and the ranks agree on the
            # outcome: a rank that cannot build must not leave its neighbours waiting in a halo exchange
            err = None
            try:
                m.prepare(batch)
            except Exception as ex:  # noqa: BLE001
                err = repr(ex)
            if parallel.max_over_ranks(0.0 if err is None else 1.0, dev) > 0:
                raise RuntimeError(err or "another rank could not build its slab plan")
            for _ in range(3):
                part = m(batch)
            ms_s, part = time_forwards(m, batch, args.steps, barrier, dev)
            X = full_logits.shape[2] // world
            mine = full_logits[:, :, rank * X:(rank + 1) * X]
            rel = float((part["ssc_logit"] - mine).abs().max() / full_logits.abs().max())
            rel = parallel.max_over_ranks(rel, dev)
            plan = list(m._plans().values())[0][0]
            xbytes = sum(getattr(op, "bytes", 0) for op in plan.ops if getattr(op, "name", "") == "halo_exchange")
            n_ex = sum(1 for op in plan.ops if getattr(op, "name", "") == "halo_exchange")
            res = {"ms_per_frame": ms_s / args.steps, "ms_per_frame_1gpu_same_run": ms_1 / args.steps,
                   "speedup_vs_1gpu": ms_1 / ms_s, "strong_scaling_efficiency": ms_1 / ms_s / world,
                   "value": N_OUT * args.steps / (ms_s * 1e-3), "unit": "voxels/s", "scaling": "strong",
                   "halo_exchanges_per_frame": n_ex, "halo_bytes_sent_per_rank_per_frame": xbytes,
                   "rel_diff_vs_unpartitioned": rel, "partition": ctx.describe() if hasattr(ctx, "describe") else
                   "X-slab of the voxel grid over %d ranks, halo 3" % world}
        except Exception as ex:  # noqa: BLE001
            res = {"error": repr(ex)}
        finally:
            m.__dict__.pop("slab_ctx", None)
            m.invalidate_plans()
    return res


_JSON_FD = None


def protect_stdout():
    """stdout carries exactly ONE JSON line: file descriptor 1 is pointed at stderr for the whole run (NCCL prints its
    version banner to stdout from C, libraries may print warnings) and the line is written to the saved descriptor."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit_json(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_JSON_FD, data)


def main():
    protect_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default=os.environ.get("OCCDEPTH_PRECISION", "tf32"), choices=["tf32", "bf16"],
                    help="arithmetic mode of the headline numbers (default: tf32, the reference-precision mode)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / cuda_reference legs")
    ap.add_argument("--no-modes", action="store_true", help="skip the second precision mode block")
    ap.add_argument("--no-slab", action="store_true", help="skip the slab block at N > 1")
    ap.add_argument("--partition", default="frames", choices=["frames", "slab"],
                    help="frames: one frame per GPU (default, weak scaling; N > 1 adds a `slab` block); slab: the "
                         "X-slab partition of one frame as the headline")
    ap.add_argument("--dump-profile", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed forward's outputs to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    run_b200(args)


if __name__ == "__main__":
    main()
