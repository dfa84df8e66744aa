#!/usr/bin/env python
"""Benchmark of the hot path (BASELINE.json: "SMPL FK+LBS meshes/s and IK frame-iters/s ...; % HBM roofline").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]

One step = one pass of the SMPL forward path (K1 pose chain + K2 fused blend-shape contraction & skinning)
over one batch of B = 4096 synthetic poses per GPU (BASELINE configs[1]); for N > 1 (torchrun, one rank per
GPU) every rank owns its own 4096 frames: frames are independent, there is no data-path collective (weak
scaling).  Rank 0 prints ONE JSON line.  The same line carries
  roofline      dominant kernel (fused blend+skinning) against the measured HBM peak, plus `lbs` for the
                standalone skinning kernel (the HBM-bound row of SURVEY.md §8d, 166 512 algorithmic B/mesh)
  e2e           the same metric through the C-ABI host-buffer call smplpp_forward_host (H2D + D2H inside)
  ik            IK frame-iterations/s of the batched MoSh step (configs[2]-shaped) when available
  cpu_baseline  the reference's own libtorch CPU implementation (oracle/_ref) on this box's host cores
`--impl reference` times only that CPU implementation and prints the line with "impl": "reference".
`--dump-outputs DIR` writes what the last timed step computed (see DUMP_FRAMES) as DIR/<name>.npy, so that two builds
can be compared output for output: the inputs are seeded and identical from run to run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 4096
VERTS = 6890
# algorithmic bytes per mesh (SURVEY.md §8d; stated in DESIGN.md)
BYTES_FUSED = VERTS * 3 * 4 + (25 * 3 + 10) * 4  # vertices out + theta, beta in
BYTES_LBS = 2 * VERTS * 3 * 4 + 24 * 12 * 4  # rest in + vertices out + 24 transforms
FLOPS_BLEND = 2 * 218 * VERTS * 3  # pose (207) + shape (10) + template (1) contraction
# --dump-outputs: vertices and joints of a fixed, seeded sample of this many frames of rank 0's batch (42 MB as float32;
# all 4096 frames would be 340 MB)
DUMP_FRAMES = 512


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_tensor_peak():
    """Dense bf16/fp16 tensor peak in TFLOP/s: the burst figure of MEASURED_PEAKS.json (a kernel timed alone), else the
    fallback of B200_PROFILING.md."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        if "bf16_tflops" in p:
            return float(p["bf16_tflops"]), "measured burst (MEASURED_PEAKS.json)"
    return 1590.0, "fallback (B200_PROFILING.md)"


def measured_tensor_peak_sustained():
    """Dense bf16 peak of a seconds-long loop under the power cap (MEASURED_PEAKS.json bf16_tflops_sustained): the
    denominator for a kernel timed inside a long step."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        if "bf16_tflops_sustained" in p:
            return float(p["bf16_tflops_sustained"]), "measured sustained (MEASURED_PEAKS.json)"
    return 1400.0, "fallback sustained (B200_PROFILING.md)"


def ncu_traffic(kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the newest committed ncu capture
    (profiles/*_traffic.json, written by scripts/ncu_summary.py); None when no capture names the kernel."""
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")), reverse=True):
        try:
            with open(path) as f:
                t = json.load(f)
            if kernel in t.get("bytes_per_launch", {}):
                return float(t["bytes_per_launch"][kernel]), os.path.basename(path)
        except Exception:
            continue
    return None, None


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                if out.returncode == 0 and out.stdout.strip():
                    self.rows.append([c.strip() for c in out.stdout.strip().split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


def cpu_reference_forward(batch_total: int, threads: int | None = None, chunk: int = 256, reps: int = 3):
    """Times the reference's own libtorch CPU forward (unmodified sources, oracle/_ref) on host cores.
    Returns (meshes/s, cores, sample description)."""
    from oracle import ref_lib
    from smplpp_b200 import synth
    if not ref_lib.available():
        raise RuntimeError("oracle/_ref/libsmplpp_ref.so is missing (built by `make -C oracle` in the build container)")
    if threads:
        ref_lib.set_num_threads(threads)
    cores = ref_lib.get_num_threads()
    ref = ref_lib.RefSMPL(ref_lib.model_json_path(0))
    beta, theta = synth.make_forward_inputs(chunk, 11)
    ref.forward(beta, theta, batched=True, want=("vertices",))  # warm-up
    best = None
    done = 0
    t_all = time.perf_counter()
    while done < batch_total:
        t0 = time.perf_counter()
        for _ in range(reps):
            ref.forward(beta, theta, batched=True, want=("vertices",))
        dt = (time.perf_counter() - t0) / reps
        best = dt if best is None else min(best, dt)
        done += chunk * reps
        if time.perf_counter() - t_all > 25:
            break
    sample = ("SMPL::launch+getVertex of the unmodified reference sources (libtorch CPU, batched build N=%d, "
              "same synthetic model/inputs), %d meshes timed" % (chunk, done))
    return chunk / best, cores, sample


def bench_config(B: int) -> dict:
    """The workload both arms (this library and `--impl reference`) are measured on: identical dict in both lines."""
    return {"workload": "configs[1]: batched SMPL forward B=%d poses/GPU fp32 (pose-blend GEMM + joint chain + LBS), "
                        "synthetic smpl_male-shaped model (6890 verts, 207 pose dims, 10 betas)" % B,
            "frames_per_gpu": B,
            "l2": "no flush: every forward pass writes %d MB of vertices (> 126 MB L2); the 18 MB blend basis is model "
                  "state that stays resident" % (B * VERTS * 12 >> 20),
            "variant": "auto"}


def run_reference(args, json_out):
    """The reference's own CPU implementation (unmodified sources, oracle/_ref) on the same config: every step is one
    pass over the B = 4096 poses (16 chunks of the batched N = 256 build), all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    B, chunk = args.batch, 256
    from oracle import ref_lib
    from smplpp_b200 import synth
    cores = os.cpu_count() or 1
    ref_lib.set_num_threads(cores)
    ref = ref_lib.RefSMPL(ref_lib.model_json_path(0))
    beta, theta = synth.make_forward_inputs(B, 11)
    nchunks = (B + chunk - 1) // chunk

    def one_pass():
        for c in range(nchunks):
            ref.forward(beta[c * chunk:(c + 1) * chunk], theta[c * chunk:(c + 1) * chunk], batched=True, want=("vertices",))

    ref.forward(beta[:chunk], theta[:chunk], batched=True, want=("vertices",))  # untimed: allocator / thread-pool warm-up
    for _ in range(max(0, min(args.warmup, 2) - 1)):
        one_pass()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one_pass()
    dt = time.perf_counter() - t0
    value = args.steps * B / dt
    line = {
        "impl": "reference", "metric": "SMPL FK+LBS meshes/s", "value": value, "unit": "meshes/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": bench_config(B),
        "cpu_baseline": {"value": value, "unit": "meshes/s", "cores": ref_lib.get_num_threads(), "kind": "reference",
                         "sample": "unmodified reference sources (oracle/_ref, libtorch CPU, batched build N=%d): one "
                                   "pass over the %d poses per step, %d steps" % (chunk, B, args.steps)},
        "e2e": {"value": value, "unit": "meshes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if not args.no_ik:
        try:
            from bench_ik import cpu_reference_ik
            v, c, sample = cpu_reference_ik(2, 2)
            line["ik"] = {"value": v, "unit": "frame-iters/s",
                          "cpu_baseline": {"value": v, "unit": "frame-iters/s", "cores": c, "kind": "reference", "sample": sample}}
            line["cpu_baseline"]["ik_value"] = v
            line["cpu_baseline"]["ik_unit"] = "frame-iters/s"
            line["cpu_baseline"]["ik_sample"] = sample
        except Exception as ex:
            line["ik"] = {"value": None, "unavailable": str(ex)}
    json_out.write(json.dumps(line) + "\n")
    json_out.flush()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH, help="frames per GPU per forward pass")
    ap.add_argument("--passes", type=int, default=160,
                    help="forward passes over the batch inside ONE timed step (a pass is 0.19 ms: 160 of them make a "
                         "step long enough for the clock sampler and the driver's consistency check)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ik", action="store_true")
    ap.add_argument("--no-config4", action="store_true", help="skip the 2^20-frame strong-scaling IK leg (BASELINE configs[4])")
    ap.add_argument("--config4-frames", type=int, default=1 << 20)
    ap.add_argument("--ik-frames-total", type=int, default=0,
                    help="BASELINE configs[4]: total mocap frames of the IK leg, sharded over the ranks as contiguous "
                         "blocks (default 0 = 16384 frames per GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the vertices and joints of the last step for a seeded sample of "
                         "%d frames as DIR/vertices.npy and DIR/joints.npy (float32)" % DUMP_FRAMES)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this library's forward pass, not of --impl reference")
    args.warmup = max(args.warmup, 3)
    # rank 0 prints ONE JSON line on stdout: libraries that write to fd 1 (NCCL's version banner) go to stderr instead
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args, json_out)

    import torch
    import torch.distributed as dist
    from smplpp_b200 import api, capi, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # one process per GPU: run on the CPUs next to it, so that the page-locked buffers of the host-buffer call and its
    # staging threads live on the GPU's NUMA node (matters once several ranks share the host)
    affinity = None
    if world > 1 and os.environ.get("SMPLPP_BENCH_NO_AFFINITY") is None:
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(local)
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
            cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
            cpus &= os.sched_getaffinity(0)
            if cpus:
                os.sched_setaffinity(0, cpus)
                affinity = len(cpus)
        except Exception:
            affinity = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    B = args.batch
    params = synth.make_smpl_params(0)
    smpl = api.SMPL(params, device=dev)
    beta_h, theta_h = synth.make_forward_inputs(B, 11 + rank)
    beta, theta = torch.as_tensor(beta_h, device=dev), torch.as_tensor(theta_h, device=dev)
    lib = capi.lib()
    import ctypes as C
    ws_bytes = lib.smplpp_forward_workspace_bytes(smpl.handle, C.c_int64(B))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    verts = torch.empty((B, VERTS, 3), dtype=torch.float32, device=dev)
    joints = torch.empty((B, 24, 3), dtype=torch.float32, device=dev)
    stream = torch.cuda.current_stream(dev)

    P = max(1, args.passes)

    def one_pass():
        capi.check(lib.smplpp_forward(smpl.handle, C.c_void_p(stream.cuda_stream), C.c_int64(B),
                                      C.c_void_p(beta.data_ptr()), C.c_int64(10), C.c_void_p(theta.data_ptr()),
                                      C.c_void_p(verts.data_ptr()), C.c_void_p(joints.data_ptr()), None, None,
                                      C.c_void_p(ws.data_ptr()), C.c_size_t(ws_bytes)))

    def step():  # one timed step = P passes of the hot path over the batch
        for _ in range(P):
            one_pass()

    # ---- the dominant kernels timed ALONE first (a few launches on a cool device: the conditions of the measured burst
    #      peaks); the same kernels inside the long headline loop run under the 1 kW power cap and are compared with
    #      the sustained peak further down ----
    def time_kernel(fn, reps):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(reps):
            fn()
        b.record(stream)
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    def k1_only():  # K1 alone = joints only
        capi.check(lib.smplpp_forward(smpl.handle, C.c_void_p(stream.cuda_stream), C.c_int64(B),
                                      C.c_void_p(beta.data_ptr()), C.c_int64(10), C.c_void_p(theta.data_ptr()),
                                      None, C.c_void_p(joints.data_ptr()), None, None, C.c_void_p(ws.data_ptr()),
                                      C.c_size_t(ws_bytes)))

    ms_k1 = time_kernel(k1_only, 20)
    ms_k2_burst = max(time_kernel(one_pass, 20) - ms_k1, 1e-6)

    for _ in range(args.warmup):
        step()
    barrier()
    launches0 = lib.smplpp_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # nvidia-smi is sampled every 100 ms from here to the end of the last measurement leg (the headline region alone is
    # steps x passes x 0.2 ms = 0.7 s with the driver's flags)
    clocks = ClockSampler(local)
    clocks.__enter__()
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    barrier()
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    launches = int(lib.smplpp_launch_count() - launches0)
    ms_step = ms_total / args.steps
    value = world * B * P / (ms_step * 1e-3)
    if args.dump_outputs and rank == 0:
        # taken now: the skinning leg below writes into `verts` again
        frames = np.sort(np.random.default_rng(0).choice(B, size=min(B, DUMP_FRAMES), replace=False))
        idx = torch.as_tensor(frames, device=dev)
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, out in (("vertices", verts), ("joints", joints)):
            np.save(os.path.join(args.dump_outputs, name + ".npy"), out.index_select(0, idx).cpu().numpy())

    # the dominant kernel inside the long loop: the step minus K1
    ms_k2 = max(ms_step / P - ms_k1, 1e-6)
    peak, peak_src = measured_peaks()
    traffic_k2, traffic_k2_src = ncu_traffic("blend_skin_tc3_kernel")
    traffic_lbs, traffic_lbs_src = ncu_traffic("lbs_tc_kernel")
    ach = BYTES_FUSED * B / (ms_k2 * 1e-3) / 1e9
    tpeak_burst, tpeak_src = measured_tensor_peak()
    tpeak, tpeak_sus_src = measured_tensor_peak_sustained()
    # The reference computes both products in fp32; on the tensor cores an fp32 product that holds the 1e-5 m tolerance
    # is THREE fp16 passes (hi.hi + lo.hi + hi.lo, fp32 accumulation): the algorithmic tensor work of the kernel is 3 x
    # (blend contraction 2.217.3V + skinning matrices 2.24.12.V) flops per mesh (DESIGN.md 4.1).
    flops_split = 3 * (2 * 217 * VERTS * 3 + 2 * 24 * 12 * VERTS) * B
    ach_t = flops_split / (ms_k2 * 1e-3) / 1e12
    roofline = {"kernel": "blend_skin_tc3_kernel (fused pose/shape blend contraction + linear blend skinning, tcgen05)",
                "bound": "tensor", "achieved": ach_t, "peak": tpeak, "unit": "TFLOP/s", "frac": ach_t / tpeak,
                "traffic": traffic_k2, "traffic_unit": "bytes per launch (dram read + write, ncu --set full)",
                "traffic_source": traffic_k2_src, "peak_source": tpeak_sus_src, "ms_per_launch": ms_k2,
                "timing": "inside the timed headline loop (%d launches back to back, power-capped): sustained peak" % (args.steps * P),
                "burst_ms_per_launch": ms_k2_burst, "burst_achieved": flops_split / (ms_k2_burst * 1e-3) / 1e12,
                "burst_peak": tpeak_burst, "burst_frac": flops_split / (ms_k2_burst * 1e-3) / 1e12 / tpeak_burst,
                "burst_peak_source": tpeak_src,
                "algorithmic_flops_per_launch": flops_split,
                "algorithmic_flops_note": "3 fp16 tensor passes per fp32 product (split precision), unpadded shapes",
                "fp32_tflops_algorithmic": FLOPS_BLEND * B / (ms_k2 * 1e-3) / 1e12,
                "algorithmic_bytes_per_launch": BYTES_FUSED * B,
                "hbm_achieved_gbs": ach, "hbm_peak_gbs": peak, "hbm_frac": ach / peak, "hbm_peak_source": peak_src}
    # the same kernel against the tensor pipe: its two products are computed as 3 fp16 passes each (hi.hi + lo.hi +
    # hi.lo, fp32 accumulation).  "split_algorithmic" counts 3 x the unpadded fp32 products (217 blend columns, 24
    # joints x 12 matrix entries), "executed" the padded tiles the MMAs really run (128 x 96 x 16 per instruction).
    tiles, fblocks = (VERTS + 127) // 128, (B + 95) // 96
    flops_exec = tiles * fblocks * (126 + 72) * (2 * 128 * 96 * 16)
    roofline["tensor"] = {"unit": "TFLOP/s", "peak": tpeak, "peak_source": tpeak_sus_src,
                          "split_algorithmic": flops_split / (ms_k2 * 1e-3) / 1e12,
                          "executed": flops_exec / (ms_k2 * 1e-3) / 1e12,
                          "frac": flops_split / (ms_k2 * 1e-3) / 1e12 / tpeak,
                          "note": "fp32 products as 3 fp16 tensor-core passes; ncu: sm__pipe_tensor_cycles_active in profiles/"}

    # standalone skinning kernel (the HBM-bound row): rest shape + 4x4 transforms -> vertices
    rest = torch.empty((B, VERTS, 3), dtype=torch.float32, device=dev)
    xf = torch.empty((B, 24, 4, 4), dtype=torch.float32, device=dev)
    capi.check(lib.smplpp_forward(smpl.handle, C.c_void_p(stream.cuda_stream), C.c_int64(B),
                                  C.c_void_p(beta.data_ptr()), C.c_int64(10), C.c_void_p(theta.data_ptr()), None, None,
                                  C.c_void_p(xf.data_ptr()), C.c_void_p(rest.data_ptr()), C.c_void_p(ws.data_ptr()),
                                  C.c_size_t(ws_bytes)))
    root = theta[:, 0].contiguous()

    xf34 = xf[:, :, :3, :].contiguous()

    def lbs_only():
        capi.check(lib.smplpp_model_skinning34(smpl.handle, C.c_void_p(stream.cuda_stream), C.c_int64(B),
                                               C.c_void_p(rest.data_ptr()), C.c_void_p(xf34.data_ptr()),
                                               C.c_void_p(root.data_ptr()), C.c_void_p(verts.data_ptr())))

    def lbs_only44():
        capi.check(lib.smplpp_model_skinning(smpl.handle, C.c_void_p(stream.cuda_stream), C.c_int64(B),
                                             C.c_void_p(rest.data_ptr()), C.c_void_p(xf.data_ptr()),
                                             C.c_void_p(root.data_ptr()), C.c_void_p(verts.data_ptr())))

    torch.cuda.synchronize()
    time.sleep(1.0)  # let the device leave the power-capped state of the headline loop: this kernel is timed alone
    ms_lbs = time_kernel(lbs_only, 20)
    ms_lbs_var = {}
    for code, name in ((200, "ffma_tma_pipeline"), (201, "ffma_register_kernel")):  # the FFMA predecessors, for comparison
        capi.check(lib.smplpp_set_forward_variant(code))
        ms_lbs_var[name] = time_kernel(lbs_only, 20)
    capi.check(lib.smplpp_set_forward_variant(202))
    ach_lbs = BYTES_LBS * B / (ms_lbs * 1e-3) / 1e9
    # flat copies (the driver keeps scalar keys of `roofline`): the HBM-bound row of SURVEY 8d
    roofline["lbs_achieved_gbs"], roofline["lbs_frac"], roofline["lbs_ms_per_launch"] = ach_lbs, ach_lbs / peak, ms_lbs
    roofline["lbs"] = {"kernel": "lbs_tc_kernel (standalone skinning, skinning matrices on tcgen05)", "bound": "hbm", "achieved": ach_lbs, "peak": peak,
                       "unit": "GB/s", "frac": ach_lbs / peak, "ms_per_launch": ms_lbs, "traffic": traffic_lbs, "traffic_source": traffic_lbs_src,
                       "algorithmic_bytes_per_launch": BYTES_LBS * B,
                       "meshes_per_s": B / (ms_lbs * 1e-3), "ms_per_launch_other_variants": ms_lbs_var,
                       "ms_per_launch_4x4_transforms": time_kernel(lbs_only44, 20)}
    del rest, xf, xf34

    # ---- e2e through the C-ABI host-buffer call: inputs in page-locked host memory, H2D + forward + D2H of the
    # vertices and joints inside the timed region (chunked two-stream pipeline, csrc/host_pipe.cu) ----
    e2e_steps = max(3, min(args.steps, 10))
    pin_beta, pin_theta = api.pinned_empty(beta_h.shape), api.pinned_empty(theta_h.shape)
    pin_beta[...], pin_theta[...] = beta_h, theta_h
    pin_v, pin_j = api.pinned_empty((B, VERTS, 3)), api.pinned_empty((B, 24, 3))
    for _ in range(2):
        smpl.launch_host(pin_beta, pin_theta, out_vertices=pin_v, out_joints=pin_j)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        smpl.launch_host(pin_beta, pin_theta, out_vertices=pin_v, out_joints=pin_j)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks((time.perf_counter() - t0) / e2e_steps)
    e2e_check = float(np.abs(pin_v[::997] - verts[::997].cpu().numpy()).max())  # same numbers as the device path
    e2e = {"value": world * B / e2e_s, "unit": "meshes/s", "h2d_bytes_per_step": int(beta_h.nbytes + theta_h.nbytes),
           "d2h_bytes_per_step": int(B * VERTS * 3 * 4 + B * 24 * 3 * 4), "ms_per_step": 1e3 * e2e_s,
           "d2h_gbs": (B * VERTS * 12 + B * 288) / e2e_s / 1e9, "max_abs_diff_vs_device_path": e2e_check,
           "api": "smplpp_forward_host (smplpp::SMPL::launch + getVertex + getRestJoint), page-locked host buffers",
           "cpu_affinity_cores": affinity}
    # the same call with ordinary pageable numpy arrays (staged through pinned chunks by host threads)
    pg_v, pg_j = np.empty((B, VERTS, 3), np.float32), np.empty((B, 24, 3), np.float32)
    smpl.launch_host(beta_h, theta_h, out_vertices=pg_v, out_joints=pg_j)
    t0 = time.perf_counter()
    for _ in range(3):
        smpl.launch_host(beta_h, theta_h, out_vertices=pg_v, out_joints=pg_j)
    e2e["pageable_value"] = world * B / max_over_ranks((time.perf_counter() - t0) / 3)
    del pg_v
    # the box's own device->host ceiling on this rank, all ranks copying at once: plain cudaMemcpyAsync of the same
    # 340 MB from device memory into the same page-locked buffer (what the link + host memory system can take)
    pin_t = torch.from_numpy(pin_v)
    for _ in range(2):
        pin_t.copy_(verts, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(5):
        pin_t.copy_(verts, non_blocking=True)
    torch.cuda.synchronize()
    d2h_s = max_over_ranks((time.perf_counter() - t0) / 5)
    e2e["d2h_ceiling_gbs"] = B * VERTS * 12 / d2h_s / 1e9
    e2e["d2h_ceiling_note"] = "per rank, all %d ranks copying concurrently; e2e d2h_gbs / ceiling = %.2f" % (
        world, e2e["d2h_gbs"] / e2e["d2h_ceiling_gbs"])
    del pin_v, pin_t

    ik = None
    if not args.no_ik:
        import bench_ik
        if args.ik_frames_total > 0:
            from smplpp_b200 import parallel
            _, nloc = parallel.frame_block(args.ik_frames_total, rank, world)
            ik = bench_ik.run(dev, rank, world, max_over_ranks, barrier, frames=nloc, iters=3, warmup=1,
                              frames_total=args.ik_frames_total)
        else:
            ik = bench_ik.run(dev, rank, world, max_over_ranks, barrier)
        if not args.no_config4:
            # BASELINE configs[4]: 2^20 frames over the N ranks (strong scaling), NCCL all-reduce of the shared-beta blocks,
            # final gather of theta
            torch.cuda.empty_cache()
            ik["config4"] = bench_ik.run_config4(dev, rank, world, max_over_ranks, barrier, frames_total=args.config4_frames)

    clocks.__exit__(None, None, None)
    line = {
        "metric": "SMPL FK+LBS meshes/s", "value": value, "unit": "meshes/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": bench_config(B),
        "passes_per_step": P, "timed_region_s": ms_total * 1e-3,
        "gpu_launches": launches, "clocks": clocks.summary(), "roofline": roofline, "e2e": e2e,
    }
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        try:
            v, cores, sample = cpu_reference_forward(1024)
            line["cpu_baseline"] = {"value": v, "unit": "meshes/s", "cores": cores, "kind": "reference", "sample": sample}
        except Exception as ex:  # the oracle library is test infrastructure; say so instead of failing the bench
            line["cpu_baseline"] = {"value": None, "unit": "meshes/s", "cores": 0, "kind": "reference",
                                    "sample": "unavailable: %s" % ex}
    if ik is not None:
        # IK is the other half of BASELINE's metric: its own roofline / e2e / cpu_baseline objects under `ik`, and flat
        # scalar copies inside the keys the driver records (nested objects are dropped from its `parsed` view)
        if rank == 0 and not args.no_cpu_baseline and world == 1:
            try:
                v, cores, sample = bench_ik.cpu_reference_ik(2, 2)
                ik["cpu_baseline"] = {"value": v, "unit": "frame-iters/s", "cores": cores, "kind": "reference", "sample": sample}
                line["cpu_baseline"].update(ik_value=v, ik_unit="frame-iters/s", ik_sample=sample)
            except Exception as ex:
                ik["cpu_baseline"] = {"value": None, "unit": "frame-iters/s", "cores": 0, "kind": "reference",
                                      "sample": "unavailable: %s" % ex}
        line["ik"] = ik
        line["ik_value"], line["ik_unit"] = ik["value"], "frame-iters/s"
        for k in ("mosh_direct", "moshpp_vposer", "shared_beta", "shared_beta_vposer"):
            if k in ik:
                line["ik_" + k] = ik[k]["value"]
        if "config4" in ik:
            c4 = ik["config4"]
            line["ik_config4_frames_total"] = c4["frames_total"]
            line["ik_config4_mosh_direct"] = c4["mosh_direct"]["value"]
            line["ik_config4_shared_beta"] = c4["shared_beta"]["value"]
            line["ik_config4_gather_s"] = c4["final_gather"]["seconds"]
        if "roofline" in ik:
            r = ik["roofline"]
            roofline.update(ik_bound=r["bound"], ik_achieved=r["achieved"], ik_peak=r["peak"], ik_unit=r["unit"],
                            ik_frac=r["frac"], ik_traffic=r.get("traffic"), ik_ms_per_iter=r.get("ms_per_launch"))
        if "e2e" in ik:
            e2e.update(ik_value=ik["e2e"]["value"], ik_unit="frame-iters/s", ik_h2d_bytes_per_step=ik["e2e"]["h2d_bytes_per_step"],
                       ik_d2h_bytes_per_step=ik["e2e"]["d2h_bytes_per_step"])
    if rank == 0:
        json_out.write(json.dumps(line) + "\n")
        json_out.flush()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
