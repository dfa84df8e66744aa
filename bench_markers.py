"""Benchmark of the markers-only forward pass (smplpp_task_forward / smplpp_task_forward_host) against the full-mesh
route it replaces (smplpp_forward + smplpp_task_positions), for the 41-marker set of synth.make_marker_tasks.

Prints ONE JSON line:
  card / power_limit_w / sm_max_mhz   read in the same run (nvidia-smi, read-only query)
  device       frames/s of smplpp_task_forward at B = 16384 and 2^20, normal offset 0 (corners only) and 0.015 (1-rings),
               and of the old route on the same inputs (at 2^20 in 16384-frame chunks: 2^20 full meshes would be 86 GB,
               plus as much forward workspace); CUDA events, warmed shapes, timed windows >= 0.5 s
  stages       per-call device time of the three kernels (chain, rest rows, task_points_kernel), from torch.profiler's
               CUDA activity records in a separate pass
  e2e          frames/s of smplpp_task_forward_host at 2^20 frames (host clock around the synchronous call), page-locked
               and pageable buffers, next to the copy ceiling of the same run: concurrent plain H2D / D2H copies of the
               same byte counts (torch non-blocking copies on two streams), and e2e as a fraction of that ceiling;
               page-locked also for several chunk sizes (SMPLPP_TASK_CHUNK)
  check        max |new - old| over a seeded 512-frame sample

usage: python bench_markers.py [--frames 1048576] [--small 16384] [--min-seconds 0.5]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import time

import numpy as np
import torch

from smplpp_b200 import api, capi, synth


def card_info():
    info = {"card": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_max_mhz": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(out[0]), float(out[1])
    except Exception:  # nvidia-smi missing: the card name alone
        pass
    return info


def time_device(fn, min_s):
    """ms per call: CUDA events around k back-to-back calls, k doubled until the window lasts >= min_s."""
    fn()
    fn()
    torch.cuda.synchronize()
    k = 1
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(k):
            fn()
        b.record()
        b.synchronize()
        ms = a.elapsed_time(b)
        if ms >= 1000 * min_s:
            return ms / k
        k *= 2


def time_host(fn, min_s):
    """ms per call of a synchronous host call (warmed), repeated until the window lasts >= min_s."""
    fn()
    k, t0 = 0, time.perf_counter()
    while True:
        fn()
        k += 1
        dt = time.perf_counter() - t0
        if dt >= min_s:
            return 1000 * dt / k


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1 << 20)
    ap.add_argument("--small", type=int, default=16384)
    ap.add_argument("--min-seconds", type=float, default=0.5)
    ap.add_argument("--chunks", default="4096,16384,65536")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    L = capi.lib()
    params = synth.make_smpl_params(0)
    smpl = api.SMPL(params, device="cuda:0")
    _, face_idx, vw = synth.make_marker_tasks(params)
    tset = api.IkTaskSet(smpl, face_idx)
    n = tset.n
    stream = api._stream(dev)
    Bbig, Bs = args.frames, args.small
    beta_h, theta_h = synth.make_forward_inputs(Bbig, 41)
    beta = torch.as_tensor(beta_h, device=dev)
    theta = torch.as_tensor(theta_h, device=dev)
    w_shared = torch.as_tensor(vw, device=dev)  # (n, 3): the MocapBody.yaml case, shared by all frames
    pos = torch.empty((Bbig, n, 3), device=dev)
    ws_new = torch.empty(L.smplpp_task_forward_workspace_bytes(tset._h, Bbig), dtype=torch.uint8, device=dev)
    # old route: one 16384-frame chunk of meshes at a time
    CH = Bs
    verts = torch.empty((CH, smpl.vertex_num, 3), device=dev)
    ws_old = torch.empty(int(L.smplpp_forward_workspace_bytes(smpl.handle, C.c_int64(CH))), dtype=torch.uint8, device=dev)
    w_rows = w_shared.expand(CH, n, 3).contiguous()
    tset.positions(verts[:1], w_rows[:1])  # uploads the face indices of the task set once

    def new_route(B, offset):
        def run():
            capi.check(L.smplpp_task_forward(smpl.handle, tset._h, stream, B, api._ptr(beta), 10, api._ptr(theta),
                                             api._ptr(w_shared), 0, offset, api._ptr(pos), None, api._ptr(ws_new),
                                             ws_new.numel()))
        return run

    def old_route(B, offset):
        def run():
            for f0 in range(0, B, CH):
                nb = min(CH, B - f0)
                capi.check(L.smplpp_forward(smpl.handle, stream, C.c_int64(nb), api._ptr(beta[f0:]), C.c_int64(10),
                                            api._ptr(theta[f0:]), api._ptr(verts), None, None, None, api._ptr(ws_old),
                                            C.c_size_t(ws_old.numel())))
                capi.check(L.smplpp_task_positions(smpl.handle, tset._h, stream, C.c_int64(nb), api._ptr(verts),
                                                   api._ptr(w_rows), C.c_float(offset), api._ptr(pos[f0:]), None))
        return run

    out = dict(metric="markers-only forward pass (41 markers): smplpp_task_forward vs smplpp_forward + smplpp_task_positions",
               **card_info(), markers=n, task_vertices=int(tset.vertex_count))
    # ---- output check (seeded 512-frame sample) ----
    check = {}
    for offset in (0.0, 0.015):
        new_route(512, offset)()
        a = pos[:512].clone()
        old_route(512, offset)()
        check["offset_%g" % offset] = float((a - pos[:512]).abs().max())
    torch.cuda.synchronize()
    out["check_max_abs_m"] = check
    # ---- device rates ----
    device = {}
    for B in (Bs, Bbig):
        for offset in (0.0, 0.015):
            key = "B%d_offset_%g" % (B, offset)
            ms_new = time_device(new_route(B, offset), args.min_seconds)
            ms_old = time_device(old_route(B, offset), args.min_seconds)
            device[key] = {"new_ms": ms_new, "new_frames_per_s": B / ms_new * 1e3, "old_ms": ms_old,
                           "old_frames_per_s": B / ms_old * 1e3, "speedup": ms_old / ms_new}
    out["device"] = device
    # ---- per-stage times (torch.profiler, separate pass) ----
    stages = {}
    from torch.profiler import ProfilerActivity, profile
    for B in (Bs, Bbig):
        for offset in (0.0, 0.015):
            run = new_route(B, offset)
            run()
            torch.cuda.synchronize()
            reps = 20 if B <= Bs else 5
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(reps):
                    run()
                torch.cuda.synchronize()
            per = {}
            for e in prof.key_averages():
                dt = getattr(e, "device_time_total", None)
                if dt is None:
                    dt = e.cuda_time_total
                if dt <= 0:
                    continue
                name = e.key.split("(")[0].split("<")[0].replace("void ", "").strip()
                per[name] = per.get(name, 0.0) + dt / 1e3 / reps
            stages["B%d_offset_%g" % (B, offset)] = {k: round(v, 5) for k, v in sorted(per.items())}
    out["stages_ms_per_call"] = stages
    # ---- end to end through host buffers at Bbig frames ----
    e2e = {}
    pin_beta, pin_theta = api.pinned_empty(beta_h.shape), api.pinned_empty(theta_h.shape)
    pin_beta[...], pin_theta[...] = beta_h, theta_h
    pin_pos = api.pinned_empty((Bbig, n, 3))
    w_np = np.ascontiguousarray(vw, dtype=np.float32)
    page_pos = np.empty((Bbig, n, 3), np.float32)

    def host_call(b, t, p, offset):
        def run():
            tset.forward_positions_host(b, t, w_np, offset, out_positions=p)
        return run

    bytes_in = Bbig * (75 + 10) * 4
    bytes_out = Bbig * n * 3 * 4
    # copy ceiling: the same byte counts as plain concurrent H2D / D2H copies
    h_in = torch.empty(bytes_in, dtype=torch.uint8).pin_memory()
    h_out = torch.empty(bytes_out, dtype=torch.uint8).pin_memory()
    d_in = torch.empty(bytes_in, dtype=torch.uint8, device=dev)
    d_out = torch.empty(bytes_out, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

    def copies():
        with torch.cuda.stream(s1):
            d_in.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_out, non_blocking=True)
        s1.synchronize()
        s2.synchronize()

    ms_ceiling = time_host(copies, args.min_seconds)
    ceiling = Bbig / ms_ceiling * 1e3
    e2e["copy_ceiling"] = {"ms": ms_ceiling, "frames_per_s": ceiling, "bytes_in": bytes_in, "bytes_out": bytes_out,
                           "GB_per_s": (bytes_in + bytes_out) / ms_ceiling / 1e6}
    default_chunk = os.environ.pop("SMPLPP_TASK_CHUNK", None)
    for label, b, t, p, offset in (("page_locked_offset_0.015", pin_beta, pin_theta, pin_pos, 0.015),
                                   ("page_locked_offset_0", pin_beta, pin_theta, pin_pos, 0.0),
                                   ("pageable_offset_0.015", beta_h, theta_h, page_pos, 0.015)):
        ms = time_host(host_call(b, t, p, offset), args.min_seconds)
        e2e[label] = {"ms": ms, "frames_per_s": Bbig / ms * 1e3, "fraction_of_copy_ceiling": ceiling and (Bbig / ms * 1e3) / ceiling}
    sweep = {}
    for ch in [int(c) for c in args.chunks.split(",") if c]:
        os.environ["SMPLPP_TASK_CHUNK"] = str(ch)
        ms = time_host(host_call(pin_beta, pin_theta, pin_pos, 0.015), args.min_seconds)
        sweep[str(ch)] = {"ms": ms, "frames_per_s": Bbig / ms * 1e3}
    os.environ.pop("SMPLPP_TASK_CHUNK", None)
    if default_chunk is not None:
        os.environ["SMPLPP_TASK_CHUNK"] = default_chunk
    e2e["page_locked_offset_0.015_by_chunk"] = sweep
    # what bounds the host entry: the device rate at the chunk size the pipeline runs vs the copy ceiling
    dev_rate = device["B%d_offset_0.015" % Bs]["new_frames_per_s"]
    e2e["bound"] = {"device_frames_per_s_at_chunk": dev_rate, "copy_ceiling_frames_per_s": ceiling,
                    "bounded_by": "device compute" if dev_rate < ceiling else "host<->device copies"}
    out["e2e"] = e2e
    # headline figures
    out["device_speedup_min"] = min(v["speedup"] for v in device.values())
    out["e2e_page_locked_frames_per_s"] = e2e["page_locked_offset_0.015"]["frames_per_s"]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
