"""Step time and binning / fine / backward phase times (CUDA events inside the library) of workloads of bench.py.

    python tools/phase_times.py [--pdl 0|1|both] ns c2 ns_blur c5 c3

(B200R_LIB=<path> times another build of the library, see pytorch3d_b200/_lib.py.)
"""
import ctypes
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from pytorch3d_b200 import _C, _lib, synthetic  # noqa: E402

args = sys.argv[1:]
pdl_modes = [1]
while args and args[0].startswith("--"):
    if args[0] == "--pdl":
        pdl_modes = [0, 1] if args[1] == "both" else [int(args[1])]
    args = args[2:]
dev = torch.device("cuda:0")
lib = _lib.load()
buf = (ctypes.c_float * 3)()


def measure(step, n_steps):
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n_steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n_steps
    lib.b200r_set_profiling(1)
    t = []
    for _ in range(min(n_steps, 12)):
        torch.cuda._sleep(400000)
        step()
        torch.cuda.synchronize()
        lib.b200r_last_phase_ms(buf)
        t.append(list(buf))
    lib.b200r_set_profiling(0)
    return ms, np.median(np.array(t[2:]), axis=0) * 1e3


for name in args or ["ns", "c2"]:
    if name == "c3":
        pc = synthetic.random_pointclouds(8, 100000, seed=0)
        pts = pc.points_packed().to(dev)
        pf, pn = pc.cloud_to_packed_first_idx().to(dev), pc.num_points_per_cloud().to(dev)
        rad = torch.full((pts.shape[0],), 0.01, device=dev)
        out = _C.rasterize_points(pts, pf, pn, (512, 512), rad, 10, 0, 0)
        gz, gd = torch.randn_like(out[1]), torch.randn_like(out[2])

        def step():
            o = _C.rasterize_points(pts, pf, pn, (512, 512), rad, 10, 0, 0)
            _C.rasterize_points_backward(pts, o[0], gz, gd)
        n_steps, hits = 30, float((out[0] >= 0).float().mean())
    else:
        nm, rings, sides, H, W, K, blur = bench.WORKLOADS[name]
        meshes = synthetic.torus_batch(nm, rings, sides, seed=0)
        fv = synthetic.face_verts_of(meshes).to(dev)
        first = meshes.mesh_to_faces_packed_first_idx().to(dev)
        num = meshes.num_faces_per_mesh().to(dev)
        nb = torch.full((fv.shape[0],), -1, dtype=torch.int64, device=dev)
        nb._b200_all_minus_one = True
        out = _C.rasterize_meshes(fv, first, num, nb, (H, W), blur, K, 0, 0, False, False, False)
        gz, gb, gd = torch.randn_like(out[1]), torch.randn_like(out[2]), torch.randn_like(out[3])

        def step():
            o = _C.rasterize_meshes(fv, first, num, nb, (H, W), blur, K, 0, 0, False, False, False)
            _C.rasterize_meshes_backward(fv, o[0], gz, gb, gd, False, False)
        n_steps, hits = (5 if name == "c5" else 40), float((out[0] >= 0).float().mean())
    for pdl in pdl_modes:
        if hasattr(lib, "b200r_set_pdl"):
            lib.b200r_set_pdl(pdl)
        ms, m = measure(step, n_steps)
        print("%-8s pdl=%d: step %.4f ms | binning %.1f us  fine %.1f us  backward %.1f us  (hits/slot %.3f)" % (
            name, pdl, ms, m[0], m[1], m[2], hits), flush=True)
    del out
