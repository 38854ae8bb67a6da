#!/usr/bin/env python
"""bench.py -- headline benchmark of the rasterizer hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path on the host cores
    python bench.py ... --dump-outputs DIR                    # + the last timed step's outputs as DIR/<name>.npy
    (N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...)

Workload ("ns", the configuration the metric is quoted on): a batch of 8 meshes of 69,938 faces each
(seeded tori in NDC), 512 x 512, faces_per_pixel = 8, blur_radius = 0, forward + backward with dense
upstream gradients on zbuf / bary / dists.  One "step" = one forward+backward pass over the batch.
Multi-GPU is weak scaling: every rank renders a batch of 8 (the SAME seeded batch on every rank, so that the
scaling figure isolates the machine; no data-path collective); `value` is frames of all ranks / max-over-ranks
device time.  The path's one collective -- gathering the rendered frames on every rank -- is timed beside it
(`value_with_gather`), and BASELINE config 4 (32 heterogeneous meshes sharded over the ranks: strong scaling)
is reported as `c4_sharded` at every N.

Prints ONE JSON line (see README / the task contract for the keys).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "rasterize frames/sec (fwd+bwd) 512^2 K=8"
UNIT = "frames/s"
WORKLOADS = {
    # name: (meshes per rank, torus rings, torus sides, H, W, K, blur)
    "ns": (8, 187, 187, 512, 512, 8, 0.0),
    "c2": (8, 54, 54, 256, 256, 8, 1e-4),
    "ns_blur": (8, 187, 187, 512, 512, 8, 1e-4),
    "ns_k16": (8, 187, 187, 512, 512, 16, 0.0),
    "c5": (1, 707, 707, 1024, 1024, 16, 1e-3),
    "tiny": (2, 24, 24, 64, 64, 4, 0.0),
}


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


NCU_SUMMARIES = ["ncu_r02_final2_ns_metrics.json", "ncu_r02_final_ns_metrics.json", "ncu_r02_ns_metrics.json", "ncu_r01_ns_metrics.json"]  # newest first


def ncu_traffic_bytes(kernel):
    """(dram read+write bytes per launch of `kernel`, source file) from the committed ncu capture summary of the
    same workload -- measured under the profiler, not in this run -- or (None, None)."""
    for name in NCU_SUMMARIES:
        path = os.path.join(ROOT, "profiles", name)
        try:
            with open(path) as fh:
                return json.load(fh)["kernels"][kernel]["dram_bytes_per_launch"], "profiles/" + name
        except Exception:
            continue
    return None, None


class ClockSampler:
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        return {
            "sm_mhz": float(np.median(self.samples)) if self.samples else None,
            "sm_max_mhz": self.max_mhz,
            "reasons": sorted(self.reasons),
            "samples": len(self.samples),
        }


# ------------------------------------------------------------------------------------------- CPU arm

def strip_transform(face_verts, y0, hs, H, W, blur):
    """Maps rows [y0, y0+hs) of an H x W render onto a full hs x W render (same pixel-face tests):
    uniform scale s = H / hs about the strip centre; squared distances (blur) scale by s^2."""
    s = float(H) / float(hs)
    fv = face_verts.clone()
    fv[..., 0] *= s
    fv[..., 1] = fv[..., 1] * s - float(H - 2 * y0 - hs) / float(hs)
    return fv, blur * s * s


def cpu_sample(face_verts, n_faces, H, W, K, blur, hs, use_ref):
    """Forward+backward of rows [y0, y0+hs) of frame 0 on the host CPU.  Returns (seconds, frames)."""
    import oracle
    fv0 = face_verts[:n_faces].contiguous()
    first = torch.zeros(1, dtype=torch.int64)
    num = torch.tensor([n_faces], dtype=torch.int64)
    y0 = (H - hs) // 2
    g = torch.Generator().manual_seed(231)
    if use_ref is not None:
        fvs, blur_s = strip_transform(fv0, y0, hs, H, W, blur)
        nb = torch.full((n_faces,), -1, dtype=torch.int64)
        t0 = time.perf_counter()
        out = use_ref.rasterize_meshes(fvs, first, num, nb, (hs, W), blur_s, K, 0, 0, False, False, False)
        gz, gb, gd = (torch.randn(o.shape, generator=g) for o in out[1:])
        use_ref.rasterize_meshes_backward(fvs, out[0], gz, gb, gd, False, False)
        dt = time.perf_counter() - t0
    else:
        fvn = fv0.numpy()
        t0 = time.perf_counter()
        out = oracle.rasterize_meshes(fvn, first.numpy(), num.numpy(), (H, W), blur, K, rows=(y0, y0 + hs))
        gz, gb, gd = (torch.randn(o.shape, generator=g).numpy() for o in out[1:])
        oracle.rasterize_meshes_backward(fvn, out[0], gz, gb, gd, rows=(y0, y0 + hs))
        dt = time.perf_counter() - t0
    return dt, float(hs) / float(H)


def load_cpu_reference():
    import oracle
    ref = oracle.load_reference(cuda=False)
    if ref is not None:
        torch.set_num_threads(os.cpu_count() or 1)
        return ref, "reference", torch.get_num_threads()
    oracle.build()
    return None, "port", os.cpu_count() or 1


def pick_strip_rows(face_verts, n_faces, H, W, K, blur, ref, budget_s, steps):
    """Calibrate on an 8-row strip, then size the strip so that `steps` samples fit in `budget_s`."""
    dt, _ = cpu_sample(face_verts, n_faces, H, W, K, blur, 8, ref)
    per_row = dt / 8.0
    rows = int(budget_s / max(steps, 1) / max(per_row, 1e-6))
    rows = max(8, min(H, (rows // 8) * 8))
    return rows


# ------------------------------------------------------------------------------------------- main

def build_workload(name, rank):
    from pytorch3d_b200 import synthetic
    nm, rings, sides, H, W, K, blur = WORKLOADS[name]
    del rank  # every rank renders the same seeded batch: per-rank seeds made the slowest rank set the time
    meshes = synthetic.torus_batch(nm, rings, sides, seed=0)
    return meshes, (nm, rings * sides * 2, H, W, K, blur)


def config_dict(name, world, nm, F1, H, W, K, blur):
    return {
        "workload": "%s: %d meshes/GPU x %d faces (seeded tori in NDC), %dx%d, faces_per_pixel=%d, "
                    "blur_radius=%g, fwd+bwd" % (name, nm, F1, H, W, K, blur),
        "meshes_per_gpu": nm, "faces_per_mesh": F1, "image_size": [H, W], "faces_per_pixel": K,
        "blur_radius": blur, "global_batch": nm * world,
        "parallelism": "batch-sharded x%d (no data-path collective; every rank renders the same seeded batch)" % world,
        "l2": "no explicit flush: each step streams ~%.0f MB of fragments + upstream gradients per GPU "
              "(>> 126 MB L2); the %.0f MB of face_verts stay L2-resident as in a real optimisation loop"
              % (nm * H * W * K * 48 / 1e6, nm * F1 * 36 / 1e6),
    }


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    name = args.workload
    meshes, (nm, F1, H, W, K, blur) = build_workload(name, 0)
    from pytorch3d_b200 import synthetic
    fv = synthetic.face_verts_of(meshes)
    ref, kind, cores = load_cpu_reference()
    rows = pick_strip_rows(fv, F1, H, W, K, blur, ref, budget_s=150.0, steps=args.steps + args.warmup)
    for _ in range(args.warmup):
        cpu_sample(fv, F1, H, W, K, blur, rows, ref)
    t_total, frames = 0.0, 0.0
    for _ in range(args.steps):
        dt, fr = cpu_sample(fv, F1, H, W, K, blur, rows, ref)
        t_total += dt
        frames += fr
    value = frames / t_total
    sample = "rows [%d,%d) of frame 0 (%d of %d rows, all %d faces) per step, fwd+bwd, %s" % (
        (H - rows) // 2, (H - rows) // 2 + rows, rows, H, F1,
        "reference C++ CPU ops (oracle/_ref/ref_raster_cpu.so, strip mapped onto a %dx%d render)" % (rows, W)
        if ref is not None else "C port (oracle/raster_oracle.c)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(name, world, nm, F1, H, W, K, blur),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


class _DeviceMeshes:
    """Packed batch whose verts/faces were just copied to the device (the e2e step's input)."""

    def __init__(self, verts, faces, first, num, max_f):
        self._v, self._f, self._first, self._num, self._F = verts, faces, first, num, max_f

    def verts_packed(self):
        return self._v

    def faces_packed(self):
        return self._f

    def mesh_to_faces_packed_first_idx(self):
        return self._first

    def num_faces_per_mesh(self):
        return self._num


def run_ours(args, rank, local_rank, world):
    import torch.distributed as dist

    from pytorch3d_b200 import _C, _lib, rasterize_meshes, synthetic

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    name = args.workload
    meshes, (nm, F1, H, W, K, blur) = build_workload(name, rank)
    fv_host = synthetic.face_verts_of(meshes)
    fv = fv_host.to(dev)
    first = meshes.mesh_to_faces_packed_first_idx().to(dev)
    num = meshes.num_faces_per_mesh().to(dev)
    nb = torch.full((fv.shape[0],), -1, dtype=torch.int64, device=dev)
    nb._b200_all_minus_one = True
    size = (H, W)

    def fwd():
        return _C.rasterize_meshes(fv, first, num, nb, size, blur, K, 0, 0, False, False, False)

    frag = fwd()
    g = torch.Generator(device=dev).manual_seed(231)
    gz = torch.randn(frag[1].shape, generator=g, device=dev)
    gb = torch.randn(frag[2].shape, generator=g, device=dev)
    gd = torch.randn(frag[3].shape, generator=g, device=dev)

    def step():
        f = fwd()
        return f, _C.rasterize_meshes_backward(fv, f[0], gz, gb, gd, False, False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---------------- device-resident throughput (value)
    for _ in range(args.warmup):
        step()
    barrier()
    launches0 = lib.b200r_kernel_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        e0.record()
        for _ in range(args.steps):
            last = None  # the previous step's outputs are released before the step allocates its own
            last = step()
        e1.record()
        barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)
    last = None
    launches = lib.b200r_kernel_launch_count() - launches0
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * nm * args.steps / (ms_max * 1e-3)

    # ---------------- per-kernel durations (roofline), same steps with phase events on the launch stream
    lib.b200r_set_profiling(1)
    import ctypes
    buf = (ctypes.c_float * 3)()
    ph = np.zeros(3)
    n_prof = max(3, min(args.steps, 20))
    for _ in range(n_prof):
        torch.cuda._sleep(400000)  # keep the GPU busy while the step's launches queue up: no launch gaps
        step()
        lib.b200r_last_phase_ms(buf)
        ph += np.array(list(buf))
    lib.b200r_set_profiling(0)
    ph /= n_prof
    peak, peak_src = measured_peak_gbs()
    slots = nm * H * W * K
    fine_bytes = 28.0 * slots + 36.0 * nm * F1            # fwd: write 28 B/slot, read face_verts once
    bwd_bytes = 28.0 * slots + 72.0 * nm * F1             # bwd: read 28 B/slot + face_verts, write grads
    fine_gbs = fine_bytes / (ph[1] * 1e-3) / 1e9 if ph[1] > 0 else 0.0
    fine_traffic, traffic_src = ncu_traffic_bytes("mesh_fine_kernel")
    bwd_traffic, _ = ncu_traffic_bytes("mesh_backward_kernel")
    bwd = {"ms": float(ph[2]), "algorithmic_bytes": bwd_bytes,
           "achieved": bwd_bytes / (ph[2] * 1e-3) / 1e9 if ph[2] > 0 else 0.0,
           "frac": (bwd_bytes / (ph[2] * 1e-3) / 1e9 / peak) if ph[2] > 0 else 0.0,
           # the kernel skips the 20 B/slot of upstream gradients of empty slots: what it really moves (ncu dram
           # bytes of the committed capture of this workload) over this run's launch time
           "traffic": bwd_traffic,
           "frac_by_dram_bytes": (bwd_traffic / (ph[2] * 1e-3) / 1e9 / peak) if (bwd_traffic and ph[2] > 0) else None}
    roofline = {
        "kernel": "mesh_fine_kernel<8>", "bound": "hbm", "achieved": fine_gbs, "peak": peak, "unit": "GB/s",
        "frac": fine_gbs / peak, "traffic": fine_traffic,
        "traffic_source": ("%s (ncu --set full capture of this workload; not measured in this run)" % traffic_src)
        if traffic_src else None,
        "algorithmic_bytes_per_launch": fine_bytes, "ms_per_launch": float(ph[1]), "peak_source": peak_src,
        "other_kernels": {
            "binning(zero+setup+scan+fill; the list sort runs inside the fine kernel)": {"ms": float(ph[0])},
            "mesh_backward_kernel": bwd,
        },
        "step": {"algorithmic_bytes": fine_bytes + bwd_bytes,
                 "achieved": (fine_bytes + bwd_bytes) * args.steps / (ms * 1e-3) / 1e9,
                 "frac": (fine_bytes + bwd_bytes) * args.steps / (ms * 1e-3) / 1e9 / peak},
    }

    # ---------------- the other single-GPU configs (device-resident; before the CUDA-graph section below)
    others, ref_cuda = None, None
    if rank == 0 and world == 1 and not args.skip_others:
        try:
            others = other_workloads(dev, lib, peak)
        except Exception as ex:
            others = {"error": str(ex)}
        try:
            ref_cuda = reference_cuda_leg(dev, fv, first, num, F1, H, W, K, blur, gz, gb, gd, nm)
        except Exception as ex:
            ref_cuda = {"error": str(ex)[:300]}
        # those workloads leave differently sized blocks in torch's caching allocator; start the end-to-end
        # section from the same allocator state as a run without them
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        # ... and their CPU-side input generation leaves OpenMP worker threads spinning for a moment; the serial
        # end-to-end mode is host-latency-bound and would be timed against them
        torch.cuda.synchronize(dev)
        time.sleep(1.0)

    # ---------------- end to end through the public API with HOST inputs (pinned) and host results
    # Every step copies its own inputs (verts + faces) from pinned host memory and returns the gradient and the
    # loss to the host.  The loop is software-pipelined two deep, like an input pipeline that prefetches the
    # next batch: the H2D copies of step i+1 run on a copy stream while step i computes, and the host reads the
    # results of step i-1 while step i runs.  All copies of all timed steps happen inside the timed region; the
    # strictly serial figure (copy -> compute -> read back -> next step) is reported next to it.
    verts_h = meshes.verts_packed().pin_memory()
    faces_h = meshes.faces_packed().pin_memory()
    max_f = int(meshes.num_faces_per_mesh().max())
    compute = torch.cuda.current_stream(dev)
    copier = torch.cuda.Stream(device=dev)
    slots = []
    for _ in range(2):
        slots.append({
            "v": torch.empty(verts_h.shape, dtype=verts_h.dtype, device=dev),
            "f": torch.empty(faces_h.shape, dtype=faces_h.dtype, device=dev),
            "grad_h": torch.empty(verts_h.shape, dtype=verts_h.dtype).pin_memory(),
            "loss_h": torch.empty((), dtype=torch.float32).pin_memory(),
            "copied": torch.cuda.Event(), "done": torch.cuda.Event(), "free": torch.cuda.Event(),
        })

    def enqueue_copy(sl):
        with torch.cuda.stream(copier):
            copier.wait_event(sl["free"])  # the previous user of this slot's device buffers has finished
            sl["v"].copy_(verts_h, non_blocking=True)
            sl["f"].copy_(faces_h, non_blocking=True)
            sl["copied"].record(copier)

    reader = torch.cuda.Stream(device=dev)  # D2H of the results: off the compute stream's critical path
    gz_flat, gb_flat, gd_flat = gz.reshape(-1), gb.reshape(-1), gd.reshape(-1)

    class _FragmentLoss(torch.autograd.Function):
        """loss = <zbuf, gz> + <bary, gb> + <dists, gd> with fixed upstream tensors: three fused dot products forward;
        backward hands d loss / d fragments = (gz, gb, gd) * grad_loss to the rasterizer.  `loss.backward()` seeds
        grad_loss with the constant 1, for which the product is the upstream tensor itself: it is passed on as is
        instead of being copied through a multiply (335 MB read + written per step for nothing)."""

        @staticmethod
        def forward(ctx, zbuf, bary, dists):
            return torch.dot(zbuf.reshape(-1), gz_flat) + torch.dot(bary.reshape(-1), gb_flat) + \
                torch.dot(dists.reshape(-1), gd_flat)

        @staticmethod
        def backward(ctx, grad_loss):
            # the benchmark only ever calls loss.backward() on this scalar: grad_loss == 1
            return gz, gb, gd

    def fragment_loss(zbuf, bary, dists):
        return _FragmentLoss.apply(zbuf, bary, dists)

    def step_body(sl):
        v = sl["v"].detach().requires_grad_(True)
        m = _DeviceMeshes(v, sl["f"], first, num, max_f)
        p2f, zbuf, bary, dists = rasterize_meshes(m, size, blur_radius=blur, faces_per_pixel=K)
        loss = fragment_loss(zbuf, bary, dists)
        loss.backward()
        sl["grad_d"], sl["loss_d"] = v.grad, loss.detach()

    def enqueue_compute(sl, overlap_d2h):
        compute.wait_event(sl["copied"])
        compute.wait_event(sl["done"])  # (graph mode: the slot's static result tensors have been read back)
        if sl.get("graph") is not None:
            sl["graph"].replay()  # the same public-API calls, captured once per slot in a CUDA graph
        else:
            step_body(sl)
        sl["free"].record(compute)
        out_stream = reader if overlap_d2h else compute
        with torch.cuda.stream(out_stream):
            out_stream.wait_event(sl["free"])
            sl["grad_h"].copy_(sl["grad_d"], non_blocking=True)
            sl["loss_h"].copy_(sl["loss_d"], non_blocking=True)
            if overlap_d2h and sl.get("graph") is None:
                sl["grad_d"].record_stream(reader)
                sl["loss_d"].record_stream(reader)
            sl["done"].record(out_stream)

    def capture_graphs():
        """The step (public API forward + loss + backward) captured in one CUDA graph per input slot: the host then
        issues one launch per step instead of ~60.  The result tensors of the capture are static; they are copied
        to the host after every replay."""
        for sl in slots:
            sl["v"].copy_(verts_h)
            sl["f"].copy_(faces_h)
        torch.cuda.synchronize(dev)
        for sl in slots:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                step_body(sl)
            sl["graph"] = g
        torch.cuda.synchronize(dev)

    def run_e2e(n, pipelined):
        out = 0.0
        for sl in slots:
            sl["free"].record(compute)
            sl["done"].record(compute)
        if not pipelined:
            for i in range(n):
                sl = slots[i & 1]
                enqueue_copy(sl)
                enqueue_compute(sl, False)
                sl["done"].synchronize()
                out += float(sl["loss_h"])
            return out
        enqueue_copy(slots[0])
        for i in range(n):
            if i + 1 < n:
                enqueue_copy(slots[(i + 1) & 1])
            enqueue_compute(slots[i & 1], True)
            if i > 0:
                slots[(i - 1) & 1]["done"].synchronize()
                out += float(slots[(i - 1) & 1]["loss_h"])
        slots[(n - 1) & 1]["done"].synchronize()
        return out + float(slots[(n - 1) & 1]["loss_h"])

    n_e2e = max(3, min(args.steps, 50))
    e2e_rates = {}

    def time_e2e(pipelined):
        run_e2e(min(args.warmup, 5) or 1, pipelined)
        torch.cuda.synchronize(dev)
        barrier()
        t0 = time.perf_counter()
        run_e2e(n_e2e, pipelined)
        torch.cuda.synchronize(dev)
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        return world * nm * n_e2e / float(dt.item())

    e2e_rates["serial"] = time_e2e(False)
    e2e_rates["pipelined"] = time_e2e(True)
    graph_note = None
    try:
        capture_graphs()
        e2e_rates["pipelined+graph"] = time_e2e(True)
    except Exception as ex:  # report, do not hide: the eager numbers above stand on their own
        graph_note = "CUDA graph capture failed: %s" % str(ex)[:200]
        for sl in slots:
            sl["graph"] = None
    for sl in slots:
        sl["graph"] = None
    best = max(e2e_rates, key=lambda k: e2e_rates[k] if k != "serial" else 0.0)
    e2e = {
        "value": e2e_rates[best], "unit": UNIT,
        "h2d_bytes_per_step": int(verts_h.numel() * 4 + faces_h.numel() * 8),
        "d2h_bytes_per_step": int(verts_h.numel() * 4 + 4),
        "steps": n_e2e, "mode": best, "modes": e2e_rates,
        "what": "pytorch3d_b200.rasterize_meshes(meshes) + loss.backward(): verts/faces H2D from pinned host "
                "memory, gradient w.r.t. verts and the loss D2H, every step; fragments stay on the device; loss = <fragments, "
                "fixed upstream> (three dot products; its backward hands the upstream tensors to the rasterizer). "
                "serial = no overlap between steps; pipelined = next step's H2D on a copy stream, results copied back on a third stream and read "
                "one step late; +graph = the step's launches replayed from a CUDA graph captured from the same "
                "public-API calls",
    }
    if graph_note:
        e2e["note"] = graph_note

    # ---------------- the same through the host-buffer C ABI (all fragments to the host)
    e2e_abi = None
    if rank == 0 and not args.skip_host_abi:
        try:
            e2e_abi = host_abi_e2e(lib, fv_host, meshes, nm, F1, H, W, K, blur)
        except Exception as ex:  # never fatal for the headline line
            e2e_abi = {"error": str(ex)}

    # ---------------- CPU baseline (rank 0, N == 1 only): bounded sample on the host cores
    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        ref, kind, cores = load_cpu_reference()
        rows = pick_strip_rows(fv_host, F1, H, W, K, blur, ref, budget_s=40.0, steps=1)
        dtc, fr = cpu_sample(fv_host, F1, H, W, K, blur, rows, ref)
        cpu = {"value": fr / dtc, "unit": UNIT, "cores": cores, "kind": kind,
               "sample": "rows [%d,%d) of frame 0 (%d of %d rows, all %d faces), fwd+bwd, %.1f s of CPU work" % (
                   (H - rows) // 2, (H - rows) // 2 + rows, rows, H, F1, dtc)}

    # ---------------- the path's one collective: every rank gathers the rendered frames of all ranks
    gather = None
    if world > 1:
        try:
            gather = gather_leg(args, dev, rank, world, nm, fwd, fv, gz, gb, gd, barrier)
        except Exception as ex:
            gather = {"error": str(ex)[:300]}
    # ---------------- BASELINE config 4: 32 heterogeneous meshes sharded over the ranks (strong scaling)
    c4 = None
    if not args.skip_c4:
        try:
            c4 = c4_leg(args, dev, rank, world, barrier)
        except Exception as ex:
            c4 = {"error": str(ex)[:300]}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(name, world, nm, F1, H, W, K, blur),
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks.summary(), "roofline": roofline,
            "cpu_baseline": cpu, "e2e_host_abi": e2e_abi, "other_workloads": others, "reference_cuda": ref_cuda,
            "value_with_gather": (gather or {}).get("value"), "with_frame_gather": gather, "c4_sharded": c4,
            "impl": "pytorch3d_b200",
        }
        print(json.dumps(line), flush=True)


DUMP_BYTES = 60 * 1000 * 1000  # what --dump-outputs may write: with the .npy headers, under 64 MB in all


def _seeded_rows(n, keep, seed=0):
    """`keep` of `n` row indices, a fixed seeded sample in ascending order (all of them when keep >= n)."""
    if keep >= n:
        return torch.arange(n)
    return torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:keep].sort().values


def dump_outputs(out_dir, frags, grad_face_verts):
    """Writes what the timed step returns -- the Fragments (pix_to_face, zbuf, bary_coords, dists) and the gradient
    w.r.t. face_verts -- as out_dir/<name>.npy in float32 (pix_to_face in float64: exact).  Each half of DUMP_BYTES
    holds one of the two; where an output does not fit, a fixed seeded sample of its pixels (all K slots) or faces is
    written, the same rows for every build, so that two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    p2f = frags[0]
    N, H, W, K = (int(v) for v in p2f.shape)
    pix = _seeded_rows(N * H * W, DUMP_BYTES // 2 // (K * (8 + 4 + 12 + 4))).to(p2f.device)
    for name, t in zip(("pix_to_face", "zbuf", "bary_coords", "dists"), frags):
        rows = t.reshape((N * H * W,) + tuple(t.shape[3:]))[pix]
        np.save(os.path.join(out_dir, name + ".npy"),
                rows.to(torch.float64 if name == "pix_to_face" else torch.float32).cpu().numpy())
    F = int(grad_face_verts.shape[0])
    faces = _seeded_rows(F, DUMP_BYTES // 2 // 36).to(grad_face_verts.device)
    np.save(os.path.join(out_dir, "grad_face_verts.npy"), grad_face_verts[faces].float().cpu().numpy())


def _time_ms(fn, steps=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def _phase_ms(lib, fn, n=5):
    """(binning, fine, backward) ms of `fn` from the library's phase events on the launch stream."""
    import ctypes
    lib.b200r_set_profiling(1)
    buf = (ctypes.c_float * 3)()
    acc = np.zeros(3)
    for _ in range(n):
        torch.cuda._sleep(400000)
        fn()
        lib.b200r_last_phase_ms(buf)
        acc += np.array(list(buf))
    lib.b200r_set_profiling(0)
    return (acc / n).tolist()


def _mesh_workload_numbers(dev, lib, peak, name, steps=20, warm=3):
    from pytorch3d_b200 import _C, synthetic
    meshes, (nm, F1, H, W, K, blur) = build_workload(name, 0)
    fv = synthetic.face_verts_of(meshes).to(dev)
    first, num = meshes.mesh_to_faces_packed_first_idx().to(dev), meshes.num_faces_per_mesh().to(dev)
    nb = torch.full((fv.shape[0],), -1, dtype=torch.int64, device=dev)
    nb._b200_all_minus_one = True
    frag = _C.rasterize_meshes(fv, first, num, nb, (H, W), blur, K, 0, 0, False, False, False)
    g = torch.Generator(device=dev).manual_seed(231)
    gz = torch.randn(frag[1].shape, generator=g, device=dev)
    gb = torch.randn(frag[2].shape, generator=g, device=dev)
    gd = torch.randn(frag[3].shape, generator=g, device=dev)
    hits = int((frag[0] >= 0).sum())
    del frag

    def step():
        f = _C.rasterize_meshes(fv, first, num, nb, (H, W), blur, K, 0, 0, False, False, False)
        _C.rasterize_meshes_backward(fv, f[0], gz, gb, gd, False, False)

    ms = _time_ms(step, steps=steps, warm=warm)
    ph = _phase_ms(lib, step, n=min(5, steps))
    slots = nm * H * W * K
    alg = 56.0 * slots + 108.0 * nm * F1
    return {"workload": "%d x %d faces, %dx%d, K=%d, blur=%g, fwd+bwd" % (nm, F1, H, W, K, blur),
            "ms_per_step": ms, "frames_per_s": nm * 1e3 / ms, "hit_slots": hits, "slots": slots,
            "phase_ms": {"binning": ph[0], "fine": ph[1], "backward": ph[2]},
            "roofline": {"bound": "hbm", "algorithmic_bytes_per_step": alg, "achieved": alg / (ms * 1e-3) / 1e9,
                         "peak": peak, "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / peak}}


def other_workloads(dev, lib, peak):
    """Device-resident fwd+bwd throughput of the other BASELINE configs that fit one GPU, and of the north-star batch
    with a blur band (context next to the metric, each with its own HBM-roofline fraction)."""
    from pytorch3d_b200 import _C, synthetic
    out = {}
    out["config2_meshes_8x5832_faces_256_K8_blur1e-4"] = _mesh_workload_numbers(dev, lib, peak, "c2")
    out["ns_blur1e-4"] = _mesh_workload_numbers(dev, lib, peak, "ns_blur")
    out["ns_K16(shared-memory queue kernel)"] = _mesh_workload_numbers(dev, lib, peak, "ns_k16")
    out["config5_1M_faces_1024_K16_blur1e-3"] = _mesh_workload_numbers(dev, lib, peak, "c5", steps=3, warm=1)
    # config 3: 8 x 100k points, 512^2, K=10, r=0.01 -- rasterization alone, then with alpha_composite (4 channels)
    pc = synthetic.random_pointclouds(8, 100000, seed=0)
    pts = pc.points_packed().to(dev)
    pf, pn = pc.cloud_to_packed_first_idx().to(dev), pc.num_points_per_cloud().to(dev)
    r = 0.01
    rad = torch.full((pts.shape[0],), r, device=dev)
    # (features_packed() is (P, C); the renderer hands its (C, P) view to the compositor, points/renderer.py:66-70)
    feats = torch.rand(pts.shape[0], 4, device=dev).permute(1, 0)
    idx, zb, d2 = _C.rasterize_points(pts, pf, pn, (512, 512), rad, 10, 0, 0)
    g_img = torch.randn(8, 4, 512, 512, device=dev)
    g_z = torch.randn_like(zb)
    g_d = torch.randn_like(d2)

    def raster_c3():
        i, z, d = _C.rasterize_points(pts, pf, pn, (512, 512), rad, 10, 0, 0)
        _C.rasterize_points_backward(pts, i, g_z, g_d)

    ms = _time_ms(raster_c3)
    ph = _phase_ms(lib, raster_c3)
    alg = 8 * (24.0 * 512 * 512 * 10 + 40.0 * 100000)
    out["config3_points_8x100k_512_K10_r0.01_raster_only"] = {
        "ms_per_step": ms, "frames_per_s": 8e3 / ms, "phase_ms": {"binning": ph[0], "fine": ph[1], "backward": ph[2]},
        "roofline": {"bound": "hbm", "algorithmic_bytes_per_step": alg, "achieved": alg / (ms * 1e-3) / 1e9,
                     "peak": peak, "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / peak}}

    def step_c3():
        i, z, d = _C.rasterize_points(pts, pf, pn, (512, 512), rad, 10, 0, 0)
        w = (1 - d / (r * r)).permute(0, 3, 1, 2)
        il = i.long().permute(0, 3, 1, 2)
        _C.accum_alphacomposite(feats, w, il)
        gf, ga = _C.accum_alphacomposite_backward(g_img, feats, w, il)
        gdd = (ga * (-1.0 / (r * r))).permute(0, 2, 3, 1).contiguous()
        _C.rasterize_points_backward(pts, i, g_z, gdd)

    ms = _time_ms(step_c3)
    out["config3_points_8x100k_512_K10_r0.01_alpha_composite"] = {
        "ms_per_step": ms, "frames_per_s": 8e3 / ms,
        "what": "rasterize_points + the reference renderer's chain (weights = 1 - d / r^2 in torch, idx.long(), permuted "
                "views, accum_alphacomposite) forward + backward"}

    def step_c3_fused():
        i, z, d = _C.rasterize_points(pts, pf, pn, (512, 512), rad, 10, 0, 0)
        _C.points_alpha_render(feats, i, d, r)
        gf, gdd = _C.points_alpha_render_backward(g_img, feats, i, d, r)
        _C.rasterize_points_backward(pts, i, g_z, gdd)

    ms = _time_ms(step_c3_fused)
    out["config3_points_8x100k_512_K10_r0.01_alpha_composite_fused"] = {
        "ms_per_step": ms, "frames_per_s": 8e3 / ms,
        "what": "rasterize_points + points_alpha_render (weights and compositing fused, on the rasterizer's own "
                "layout) forward + backward; same images bit for bit"}
    return out


def reference_cuda_leg(dev, fv, first, num, F1, H, W, K, blur, gz, gb, gd, nm):
    """The reference's own CUDA kernels rebuilt for sm_100a (oracle/_ref/ref_raster_cuda.so) on the same GPU and
    batch, with the reference's default heuristics (rasterize_meshes.py:122-142): the bar SURVEY.md 2.2 names.
    Timed outside every timed region of `value`."""
    import oracle
    ref = oracle.load_reference(cuda=True)
    if ref is None:
        return {"unavailable": "oracle/_ref/ref_raster_cuda.so not present on this box"}
    size = max(H, W)
    bin_size = 8 if size <= 64 else int(2 ** max(np.ceil(np.log2(size)) - 4, 4))
    max_faces_per_bin = int(max(10000, F1 / 5))
    nb = torch.full((fv.shape[0],), -1, dtype=torch.int64, device=dev)

    def fwd():
        return ref.rasterize_meshes(fv, first, num, nb, (H, W), blur, K, bin_size, max_faces_per_bin, False, False,
                                    False)

    frag = fwd()
    t_f = _time_ms(fwd, steps=3, warm=1)
    t_b = _time_ms(lambda: ref.rasterize_meshes_backward(fv, frag[0], gz, gb, gd, False, False), steps=3, warm=1)
    return {"fwd_ms": t_f, "bwd_ms": t_b, "frames_per_s": nm * 1e3 / (t_f + t_b), "bin_size": bin_size,
            "max_faces_per_bin": max_faces_per_bin,
            "what": "pytorch3d/csrc/rasterize_{coarse,meshes}/*.cu compiled unmodified for sm_100a, coarse-to-fine, "
                    "same batch, same GPU, CUDA events, 3 repeats"}


def gather_leg(args, dev, rank, world, nm, fwd, fv, gz, gb, gd, barrier):
    """The step with every rank receiving the frames of all ranks, off the critical path: the exchange of step i
    overlaps the backward pass of step i and the forward pass of step i+1 (at most two exchanges in flight).
    Two transports: `nccl_dense` = 4 x all_gather_into_tensor with pix_to_face narrowed to int32 on the wire;
    `peer_packed` = one kernel packs the valid slots (1 B per pixel + 24 B per hit) and stores them straight into
    every peer's memory over NVLink, one kernel per source expands them (pytorch3d_b200/peer.py)."""
    import torch.distributed as dist

    from pytorch3d_b200 import _C, parallel, peer
    N = nm * world
    plan = parallel.ShardPlan([list(range(r * nm, (r + 1) * nm)) for r in range(world)],
                              [0] * N, [0] * N)
    f0 = fwd()
    K = int(f0[0].shape[-1])
    H, W = int(f0[0].shape[1]), int(f0[0].shape[2])
    slots = f0[0].numel()
    hits = int((f0[0] >= 0).sum())
    n_g = max(3, min(args.steps, 20))

    def timed(start):
        def run(n):
            prev = None
            for _ in range(n):
                f = fwd()
                h = start(f)
                _C.rasterize_meshes_backward(fv, f[0], gz, gb, gd, False, False)
                if prev is not None:
                    prev.wait()
                prev = h
            prev.wait()
        run(3)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        run(n_g)
        g1.record()
        barrier()
        tg = torch.tensor([g0.elapsed_time(g1)], dtype=torch.float64, device=dev)
        dist.all_reduce(tg, op=dist.ReduceOp.MAX)
        return float(tg.item()) / n_g

    out = {"unit": UNIT, "steps": n_g,
           "what": "fwd -> [exchange of this step's frames, on a side stream] overlapped with bwd and the next fwd; "
                   "every rank ends up with all Fragments (int64 pix_to_face, zbuf, bary, dists) of all ranks"}
    fg = parallel.FrameGather(plan, rank)
    ms = timed(fg.start)
    wire = slots * 24 * (world - 1)
    out["nccl_dense"] = {"value": N / (ms * 1e-3), "ms_per_step": ms, "bytes_received_per_rank_per_step": int(wire),
                         "receive_gb_per_s_per_rank": wire / (ms * 1e-3) / 1e9,
                         "limit": "NVLink ingress of every rank: (N-1)/N of all frames at 24 B per (pixel, slot) "
                                  "against 770 GB/s measured peer bandwidth per direction (900 nominal)"}
    try:
        ex = peer.PackedFrameExchange(plan, rank, (H, W), K)
        try:
            ms_p = timed(ex.start)
        finally:
            ex.close()
        wire_p = (slots // K + hits * 24) * (world - 1)
        dense_out = slots * 28 * (world - 1)
        out["peer_packed"] = {
            "value": N / (ms_p * 1e-3), "ms_per_step": ms_p, "bytes_received_per_rank_per_step": int(wire_p),
            "receive_gb_per_s_per_rank": wire_p / (ms_p * 1e-3) / 1e9, "valid_slot_fraction": hits / slots,
            "dense_bytes_expanded_per_rank_per_step": int(dense_out),
            "limit": "HBM writes of the expansion: (N-1)/N of all frames at 28 B per (pixel, slot) into local memory "
                     "(%.2f GB per step), sharing the memory system with the rasterizer" % (dense_out / 1e9)}
    except Exception as ex_:
        out["peer_packed"] = {"error": str(ex_)[:300]}
    best = max((k for k in ("nccl_dense", "peer_packed") if "value" in out.get(k, {})),
               key=lambda k: out[k]["value"])
    out["value"], out["transport"], out["ms_per_step"] = out[best]["value"], best, out[best]["ms_per_step"]
    return out


def c4_face_counts(n=32, seed=0):
    """BASELINE config 4: face counts log-uniform in [5k, 100k] (SURVEY.md 8d)."""
    g = torch.Generator().manual_seed(seed)
    u = torch.rand(n, generator=g)
    return [int(v) for v in torch.exp(np.log(5e3) + u * (np.log(1e5) - np.log(5e3)))]


def c4_leg(args, dev, rank, world, barrier):
    """BASELINE config 4: heterogeneous batch of 32 meshes (5k-100k faces), 512^2, K=8, forward+backward, sharded over
    the ranks by parallel.ShardPlan (greedy LPT on face counts); total work fixed -> strong scaling."""
    import torch.distributed as dist

    from pytorch3d_b200 import _C, parallel, synthetic
    meshes = synthetic.torus_batch_hetero(c4_face_counts(), seed=0)
    fv_all = synthetic.face_verts_of(meshes).to(dev)
    first, num = meshes.mesh_to_faces_packed_first_idx(), meshes.num_faces_per_mesh()
    plan = parallel.ShardPlan.build(first.tolist(), num.tolist(), world)
    loc = plan.local_inputs(fv_all, rank)
    del fv_all
    H = W = 512
    K = 8
    nb = torch.full((loc.face_verts.shape[0],), -1, dtype=torch.int64, device=dev)
    nb._b200_all_minus_one = True
    n_loc = len(loc.mesh_ids)
    g = torch.Generator(device=dev).manual_seed(231)
    gz = torch.randn((n_loc, H, W, K), generator=g, device=dev)
    gb = torch.randn((n_loc, H, W, K, 3), generator=g, device=dev)
    gd = torch.randn((n_loc, H, W, K), generator=g, device=dev)
    ex = None  # the frame exchange: packed, through peer memory (falls back to the dense NCCL gather)
    if world > 1:
        try:
            from pytorch3d_b200 import peer
            ex = peer.PackedFrameExchange(plan, rank, (H, W), K)
        except Exception:
            ex = None
    fg = parallel.FrameGather(plan, rank)

    def step(gather):
        f = _C.rasterize_meshes(loc.face_verts, loc.first, loc.num, nb, (H, W), 0.0, K, 0, 0, False, False, False)
        h = None
        if gather:
            h = ex.start(f) if ex is not None else fg.start([plan.rebase(f[0], rank), f[1], f[2], f[3]])
        _C.rasterize_meshes_backward(loc.face_verts, f[0], gz, gb, gd, False, False)
        return h

    def timed(gather, n):
        for _ in range(3):
            h = step(gather)
            if h is not None:
                h.wait()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        prev = None
        for _ in range(n):
            h = step(gather)
            if prev is not None:
                prev.wait()
            prev = h
        if prev is not None:
            prev.wait()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / n

    n = max(3, min(args.steps, 20))
    ms = timed(False, n)
    out = {"workload": "32 tori, faces log-uniform 5k-100k (total %d), 512x512, K=8, blur 0, fwd+bwd" % int(num.sum()),
           "scaling": "strong", "n_gpus": world, "ms_per_step": ms, "frames_per_s": 32e3 / ms,
           "faces_per_rank": [int(sum(plan.num[i] for i in ids)) for ids in plan.assignment],
           "meshes_per_rank": [len(ids) for ids in plan.assignment]}
    if world > 1:
        ms_g = timed(True, n)
        out["with_frame_gather"] = {"ms_per_step": ms_g, "frames_per_s": 32e3 / ms_g,
                                    "transport": "peer_packed" if ex is not None else "nccl_dense"}
        if ex is not None:
            ex.close()
    return out


def host_abi_e2e(lib, fv_host, meshes, nm, F1, H, W, K, blur, steps=3):
    """forward_host + backward_host of the C ABI: every buffer is host memory (pinned)."""
    slots = nm * H * W * K
    fv = fv_host.contiguous().pin_memory()
    first = meshes.mesh_to_faces_packed_first_idx().pin_memory()
    num = meshes.num_faces_per_mesh().pin_memory()
    p2f = torch.empty(slots, dtype=torch.int64).pin_memory()
    z = torch.empty(slots, dtype=torch.float32).pin_memory()
    b = torch.empty(slots * 3, dtype=torch.float32).pin_memory()
    d = torch.empty(slots, dtype=torch.float32).pin_memory()
    g = torch.Generator().manual_seed(231)
    gz = torch.randn(slots, generator=g).pin_memory()
    gb = torch.randn(slots * 3, generator=g).pin_memory()
    gd = torch.randn(slots, generator=g).pin_memory()
    out = torch.empty_like(fv).pin_memory()
    F = fv.shape[0]

    def once():
        rc = lib.b200r_rasterize_meshes_forward_host(fv.data_ptr(), F, first.data_ptr(), num.data_ptr(), None, nm, H,
                                                     W, blur, K, 0, 0, 0, p2f.data_ptr(), z.data_ptr(), b.data_ptr(),
                                                     d.data_ptr())
        assert rc == 0, lib.b200r_last_error()
        rc = lib.b200r_rasterize_meshes_backward_host(fv.data_ptr(), F, p2f.data_ptr(), gz.data_ptr(), gb.data_ptr(),
                                                      gd.data_ptr(), nm, H, W, K, 0, 0, out.data_ptr())
        assert rc == 0, lib.b200r_last_error()

    once()
    t0 = time.perf_counter()
    for _ in range(steps):
        once()
    dt = time.perf_counter() - t0
    return {"value": nm * steps / dt, "unit": UNIT, "steps": steps,
            "h2d_bytes_per_step": int(F * 36 * 2 + nm * 16 + slots * (8 + 20)),
            "d2h_bytes_per_step": int(slots * 28 + F * 36),
            "what": "b200r_rasterize_meshes_forward_host + _backward_host: all Fragments returned to host memory and "
                    "all upstream gradients read from host memory (PCIe-bound)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="ns", choices=sorted(WORKLOADS))
    ap.add_argument("--skip-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--skip-host-abi", action="store_true")
    ap.add_argument("--skip-others", action="store_true", help="skip the other configs / reference-CUDA legs")
    ap.add_argument("--skip-c4", action="store_true", help="skip the sharded config-4 leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank, local_rank, world = env_int("RANK", 0), env_int("LOCAL_RANK", 0), env_int("WORLD_SIZE", 1)
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, local_rank, world)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
