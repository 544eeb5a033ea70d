#!/usr/bin/env python3
"""bench.py — Msamples/s (and Mrays/s) of the radiance loop on BASELINE.json's configurations.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C2] [--also C3,C4,C5] [--impl ptb|reference] [--dump-outputs DIR]

A step is one full render of the named configuration (default C2 = BASELINE.json configs[1]: 1,000,000-triangle
Phong mesh + HDR-style envmap, 1024x1024, 256 spp, depth 5) on synthetic, closed-form inputs.  Scene generation,
BVH build and upload happen once before the timed region and are reported separately (SURVEY.md §8d).
  value   whole-job Msamples/s with the scene resident in HBM and the frame left in HBM (ptb_render_sharded, no host outputs)
  e2e     the same through the reference-shaped call Raytracer::render_image_nopreviz() with HOST buffers:
          camera + parameters go host->device, imagedouble + sample_count + 8-bit image come back every step
  roofline  the kernel with the largest share of the step (closest-hit BVH8 traversal on C2/C3/C5, the MERL shade kernel on C4):
          algorithmic bytes / launch time against the measured HBM copy bandwidth (the contract's formula), and next to it what
          actually bounds these kernels: instruction issue under divergence (`bound`, `issue_frac` from the committed ncu capture)
  cpu_baseline  the reference's own CPU code (oracle/_ref) or its C restatement (oracle/port) on this box's cores
  also    short measurements of the other BASELINE configurations in the same run (C3: the 2.5M-triangle target of north_star,
          C4, C5: the 24M-triangle scene the tile split is quoted on), each at its FULL resolution and spp
For N > 1 (torchrun, one rank per GPU) the frame is tile-sharded and gathered once over NCCL inside the library
(ptb_render_sharded); value = samples of all ranks / max-over-ranks time: strong scaling on the fixed frame.
`--impl reference` times the reference's CPU implementation on a FIXED number of samples per pixel per step (REF_SPP below),
whatever --steps / --warmup are, so that this arm and `cpu_baseline` measure the same thing.
`--dump-outputs DIR` writes the frame the last timed step of the named workload computed (see dump_outputs) as DIR/<name>.npy,
so that two builds can be compared output for output: the scenes are closed-form and the seed is fixed, so the inputs are identical
from run to run.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

WORKLOADS = {
    "C1": "default parametric scene (spheres + spherical light, Phong) 512x512, 64 spp, depth 5",
    "C2": "synthetic 1M-triangle diffuse/Phong mesh + envmap, 1024x1024, 256 spp, depth 5",
    "C3": "synthetic 2.5M-triangle fully transparent mesh (Fresnel) + normal/alpha maps, 1920x1080, 512 spp, depth 5",
    "C4": "synthetic MERL-format BRDF (90x90x180) on a 260k-triangle mesh with DoF, 1024x1024, 1024 spp, depth 5",
    "C5": "synthetic 24M-triangle scene, 3840x2160, 1024 spp, depth 5",
}
# Samples per pixel of one CPU step (full resolution).  The reference pays a fixed cost per render_image_nopreviz() call (one
# full-frame buffer per thread allocated, zeroed and merged serially, Raytracer.cpp:1576-1579, 1669-1685: about 0.4 s on C2 with
# 16 threads), so its Msamples/s GROWS with spp; these values are above BASELINE.md §3's plan (C2 8, C3 4, C4 8, C5 1) to keep that
# cost below ~10-20 % of a step while a step stays a few seconds.  The same value is used by `cpu_baseline` and `--impl reference`.
REF_SPP = {"C1": 64, "C2": 32, "C3": 8, "C4": 16, "C5": 2}
# algorithmic bytes per item of the kernels other than the traversals (DESIGN.md section 5)
SHADE_BYTES = 340      # queue 4 + hit/ray o/ray d/weight/radiance 80 + rng 8 + pixel 4 + TriUV 32 + TriShade 80 + rpp 8 read; ray, weight, hit 64 + rng 8 + queue 4 + shadow entry 48 written
KERNEL_LABEL = {"extend": "k_trace<closest-hit> (BVH8 traversal)", "shadow": "k_trace<any-hit> (BVH8 traversal, shadow rays)",
                "shade": "k_shade (material fetch, BRDF eval / sampling, next-event estimation)", "raygen": "k_raygen", "splat": "k_splat"}
DUMP_BYTES = 60 * 10 ** 6      # --dump-outputs stays below 64 MB with the .npy headers


def dump_outputs(rt, out_dir):
    """The frame the last timed step of `value` left on the device, resolved (ptb_resolve_last) into the arrays
    Raytracer::render_image_nopreviz() hands its caller, as float32 .npy files: the linear image (imagedouble), the per-pixel filter
    weight sums (sample_count) and the 8-bit display image (image).  A frame larger than
    DUMP_BYTES (C5) is cut down to the same seeded sample of pixels in every run; pixel_index.npy lists them (row-major)."""
    arrays = {k: np.asarray(getattr(rt, k), np.float32) for k in ("imagedouble", "sample_count", "image")}
    if sum(a.nbytes for a in arrays.values()) > DUMP_BYTES:
        n_px = rt.H * rt.W
        per_px = sum(a.nbytes for a in arrays.values()) // n_px
        idx = np.sort(np.random.default_rng(0).choice(n_px, DUMP_BYTES // (per_px + 8), replace=False))
        arrays = {k: a.reshape(n_px, *a.shape[2:])[idx] for k, a in arrays.items()}
        arrays["pixel_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # "under load": samples in the upper half of the power draw seen
        thr = 0.5 * max(pw)
        load = [s for s, p in zip(sm, pw) if p >= thr] or sm
        return {"sm_mhz": statistics.median(load), "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm), "reasons": sorted(reasons)}


def make_rt(lib, workload, device=0):
    from pathtracer_b200 import scenes
    return scenes.CONFIGS[workload](lib, device=device)


def cpu_reference(workload, steps, warmup):
    """The reference's own CPU implementation of the path on the host cores: oracle/_ref if it is here, else oracle/port.
    Every step renders the full-resolution frame at REF_SPP[workload] samples per pixel."""
    from oracles import port_lib, ref_lib
    from pathtracer_b200 import _abi
    lib = ref_lib()
    kind = "reference"
    if lib is None:
        lib, kind = port_lib(), "port"
    cores = min(os.cpu_count() or 1, 64)       # the reference is hard-limited to 64 threads (Vector.h:29, Raytracer.h:114)
    rt = make_rt(lib, workload)
    full_spp = rt.nrays
    t0 = time.time()
    rt.commit()
    build_s = time.time() - t0
    rt.set_option(_abi.ORC_OPT_THREADS, cores)
    spp = min(full_spp, REF_SPP[workload])
    rt.nrays = spp
    times, rays = [], 0
    for i in range(max(1, steps) + max(0, warmup)):
        t0 = time.time(); rt.render_image_nopreviz(want_image=False); dt = time.time() - t0
        if i >= warmup:
            times.append(dt); rays = rt.stats["rays_closest"] + rt.stats["rays_shadow"]
    samples = rt.W * rt.H * spp
    ms = 1e3 * sum(times) / len(times)
    value = samples / ms / 1e3
    base = {"value": value, "unit": "Msamples/s", "cores": cores, "kind": kind,
            "sample": f"{workload} at full resolution {rt.W}x{rt.H}, {spp} spp of {full_spp} per step (fixed, independent of --steps), depth {rt.nb_bounces}, "
                      f"{len(times)} timed step(s) after {warmup} warm-up; BVH build {build_s:.1f}s excluded",
            "mrays_per_s": rays / ms / 1e3}
    rt.close()
    return base, ms, spp


def ncu_record(workload, kernel):
    """Counters of the committed ncu --set full capture of `kernel` on `workload` (profiles/roofline_traffic.json), or {}."""
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if not os.path.exists(tpath):
        return {}
    rec = json.load(open(tpath)).get(workload, {})
    if kernel in rec and isinstance(rec[kernel], dict):
        return rec[kernel]
    return rec if kernel == "extend" else {}


def roofline(workload, kt, n_node, n_tri, serial_ms):
    """The contract's roofline object for the kernel with the largest share of the (serialised) step."""
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    step_kernel_ms = sum(v["ms"] for v in kt.values())
    top = max(kt, key=lambda k: kt[k]["ms"])
    k = kt[top]
    if top in ("extend", "shadow"):
        nn, nt = n_node[top], n_tri[top]
        bytes_per_item = 80 * nn + 48 * nt + (48 if top == "extend" else 80)
    elif top == "shade":
        nn = nt = None
        bytes_per_item = SHADE_BYTES
    else:
        nn = nt = None
        bytes_per_item = 108 if top == "raygen" else 160
    launch_ms = k["ms"] / max(1, k["launches"])
    items_per_launch = k["items"] / max(1, k["launches"])
    achieved = items_per_launch * bytes_per_item / (launch_ms * 1e-3) / 1e9 if launch_ms > 0 else 0.0
    rec = ncu_record(workload, top)
    traffic = rec.get("dram_bytes_per_launch", rec.get("k_trace_closest_dram_bytes_per_launch"))
    ncu = {q: rec[q] for q in ("issue_active_pct", "active_lanes_per_instruction", "fma_pipe_active_pct", "alu_pipe_active_pct", "dram_throughput_pct",
                               "l2_throughput_pct", "l1_hit_pct", "l2_hit_pct", "source") if q in rec} or None
    issue_frac = None
    if ncu and "issue_active_pct" in ncu and "active_lanes_per_instruction" in ncu:
        issue_frac = ncu["issue_active_pct"] / 100.0 * ncu["active_lanes_per_instruction"] / 32.0
    return {
        # `bound`: what the counters say limits the kernel.  All kernels of this path are bound by instruction issue under SIMT
        # divergence (issue-active 57-72 %, 13-25 of 32 lanes per instruction, DRAM throughput 5-30 %), not by HBM; `achieved` /
        # `peak` / `frac` are the contract's algorithmic-bytes figure against the measured HBM copy bandwidth, `issue_frac` =
        # issue-active x active lanes / 32 is the fraction of the SMs' lane-issue capacity doing useful work.
        "bound": "issue", "kernel": KERNEL_LABEL[top], "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
        "issue_frac": issue_frac, "peak_source": peak_src, "ncu": ncu, "bytes_per_item": bytes_per_item, "n_node": nn, "n_tri": nt,
        "items_per_launch": items_per_launch, "launch_ms": launch_ms, "launches_per_step": k["launches"],
        "share_of_step": k["ms"] / step_kernel_ms if step_kernel_ms else None,
        "timing": "CUDA events around every launch of one extra step with the pass pipelines serialised (PTB_OPT_PIPES=1), taken right after the timed region",
        "serialised_step_ms": serial_ms,
        "kernel_ms_per_step": {q: v["ms"] for q, v in kt.items()},
        "traversal_per_ray": {"closest": {"n_node": n_node["extend"], "n_tri": n_tri["extend"]}, "any_hit": {"n_node": n_node["shadow"], "n_tri": n_tri["shadow"]}}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="C2", choices=sorted(WORKLOADS))
    ap.add_argument("--also", default=None, help="comma-separated workloads measured briefly in the same run (default: C3,C4,C5 next to C2; '' for none)")
    ap.add_argument("--impl", default="ptb", choices=["ptb", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of --workload as DIR/<name>.npy (float32, under 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; --impl reference renders fewer spp than the workload")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    also = args.also if args.also is not None else ("C3,C4,C5" if args.workload == "C2" else "")
    also = [w for w in also.split(",") if w and w != args.workload]
    base_line = {"metric": "Msamples/s", "unit": "Msamples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                 "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                 "config": {"workload": f"{args.workload}: {WORKLOADS[args.workload]}", "spp_sharding": "image tiles (32x32 when shared, 16x16 among 8 GPUs, rows rotated), tile_id % n_gpus",
                            "pass_pipelines": int(os.environ.get("PTB_PIPES", "2")),
                            "l2": "working set per step (BVH + triangles + path pool, >2 GB) exceeds the 126 MB L2; no flush needed"}}

    if args.impl == "reference":
        if rank != 0:
            return 0
        cb, ms, spp = cpu_reference(args.workload, args.steps, args.warmup)
        line = dict(base_line)
        line.update({"impl": "reference", "value": cb["value"], "ms_per_step": ms, "n_gpus": args.gpus, "cpu_baseline": cb,
                     "e2e": {"value": cb["value"], "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0})
        print(json.dumps(line), flush=True)
        return 0

    import torch
    import torch.distributed as dist
    import pathtracer_b200
    from pathtracer_b200 import _abi, multi
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    lib = pathtracer_b200.load()
    N_PIPES = int(os.environ.get("PTB_PIPES", "2"))

    def sync():
        torch.cuda.synchronize(device)
        if world > 1:
            dist.barrier()

    def measure(workload, steps, warmup, brief, dump_dir=None):
        """One workload on this rank's GPU.  brief: the warm-up steps and the instrumented steps run at reduced spp (they warm clocks and
        allocations and time single launches, which do not depend on the number of passes); the timed steps are always full renders.
        dump_dir: where rank 0 writes the outputs of the last timed step (dump_outputs)."""
        t0 = time.time(); rt = make_rt(lib, workload, device=local); gen_s = time.time() - t0
        rt.build_threads = max(1, (os.cpu_count() or 1) // max(1, world))   # torchrun exports OMP_NUM_THREADS=1
        t0 = time.time(); rt.commit(); commit_s = time.time() - t0
        rt.reuse_buffers = True     # like the reference, whose Raytracer owns its output vectors (Raytracer.h:90-105)
        multi.init_comm(rt, rank, world)
        info = rt.scene_info()
        full_spp = rt.nrays
        samples_frame = rt.W * rt.H * full_spp
        spp_pool = max(1, (1 << 25) // (rt.W * rt.H))
        short_spp = min(full_spp, max(8, 8 * spp_pool)) if brief else full_spp

        def timed(fn, k):
            sync()
            t0 = time.perf_counter()
            dev_ms, launches, rays = 0.0, 0, 0
            for _ in range(k):
                fn()
                st = rt.stats
                dev_ms += st["ms_device"]; launches += st["kernel_launches"]; rays += st["rays_closest"] + st["rays_shadow"]
            sync()
            wall_ms = 1e3 * (time.perf_counter() - t0)
            t = torch.tensor([wall_ms, dev_ms], dtype=torch.float64, device=device)
            tot = torch.tensor([launches, rays], dtype=torch.int64, device=device)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dist.all_reduce(tot, op=dist.ReduceOp.SUM)
            return float(t[0]), float(t[1]), int(tot[0]), int(tot[1])

        # instrumented, untimed pass: traversal counters for the roofline's algorithmic bytes (same kernels, same config)
        rt.set_option(_abi.OPT_COUNT_TRAVERSAL, 1)
        rt.nrays = min(full_spp, 8)
        rt.render_resident()
        kt = rt.kernel_times()
        n_node = {k: kt[k]["node_visits"] / max(1, kt[k]["items"]) for k in ("extend", "shadow")}
        n_tri = {k: kt[k]["tri_tests"] / max(1, kt[k]["items"]) for k in ("extend", "shadow")}
        rt.set_option(_abi.OPT_COUNT_TRAVERSAL, 0)

        rt.nrays = short_spp
        t_w = time.perf_counter()
        for _ in range(warmup):
            rt.render_resident()
        if brief:
            # A sharded short-spp step is a few tens of ms: two of them after a multi-second BVH build leave the clocks below boost
            # and the first timed step pays for it (r02m: C3 at N=8 193 ms per step against 157 ms through the host route measured
            # right after).  Warm up for at least a second, then time enough full steps for about two seconds of rendering.
            n_w = warmup
            while True:
                el = torch.tensor([time.perf_counter() - t_w], dtype=torch.float64, device=device)
                if world > 1:
                    dist.all_reduce(el, op=dist.ReduceOp.MAX)
                if float(el[0]) >= 1.0 or n_w >= 64:
                    break
                rt.render_resident(); n_w += 1
            warmup = n_w
            sync(); t1 = time.perf_counter(); rt.render_resident(); sync()
            est = torch.tensor([(time.perf_counter() - t1) * full_spp / short_spp], dtype=torch.float64, device=device)
            if world > 1:
                dist.all_reduce(est, op=dist.ReduceOp.MAX)
            steps = max(steps, min(6, int(2.0 / max(float(est[0]), 1e-3))))
        rt.nrays = full_spp
        if brief and world > 1:
            # the first full-spp sharded step after short ones ran 8 % (C3) to 20 % (C5) slower than the ones after it at N = 8
            # (profiles/r02aa: `value` below `e2e`, which is measured later in the same process): one untimed full step first
            rt.render_resident()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        wall_ms, dev_ms, launches, rays = timed(rt.render_resident, steps)
        if dump_dir and rank == 0:
            rt.resolve_last()          # the frame the last timed step left on the device
            dump_outputs(rt, dump_dir)
        # per-kernel CUDA-event timing (two event records per launch on the launching stream).  The timed region above runs the passes
        # on two pipelines (streams) whose kernels overlap, so a kernel's own duration is taken from one more step of the same
        # workload, right here, with the pipelines serialised: `roofline.launch_ms` is the kernel running alone on the GPU.
        rt.set_option(_abi.OPT_PIPES, 1)
        rt.set_option(_abi.OPT_TIME_KERNELS, 1)
        rt.nrays = short_spp
        rt.render_resident()
        kt = rt.kernel_times()
        scale = full_spp / short_spp
        for v in kt.values():          # per full step
            v["ms"] *= scale; v["launches"] = int(round(v["launches"] * scale)); v["items"] = int(round(v["items"] * scale))
        serial_ms = rt.stats["ms_device"] * scale
        rt.set_option(_abi.OPT_TIME_KERNELS, 0)
        rt.set_option(_abi.OPT_PIPES, N_PIPES)
        rt.nrays = short_spp       # one untimed call through the host-buffer route (its output arrays get allocated and page-locked here)
        rt.render_image_nopreviz(want_image=True)
        rt.nrays = full_spp
        e2e_ms, _, _, _ = timed(lambda: rt.render_image_nopreviz(want_image=True), steps)
        clocks = sampler.stop() if rank == 0 else None

        ms_per_step = wall_ms / steps
        res = {"value": samples_frame / ms_per_step / 1e3, "ms_per_step": ms_per_step, "device_ms_per_step": dev_ms / steps,
               "mrays_per_s": rays / steps / ms_per_step / 1e3, "rays_per_sample": rays / steps / samples_frame,
               "gpu_launches": launches, "clocks": clocks,
               "e2e": {"value": samples_frame / (e2e_ms / steps) / 1e3, "unit": "Msamples/s",
                       "h2d_bytes_per_step": C.sizeof(_abi.Camera) + C.sizeof(_abi.Params), "d2h_bytes_per_step": rt.W * rt.H * (12 + 4 + 3)},
               "setup": {"scene_gen_s": gen_s, "commit_s": commit_s, "bvh_build_ms": info["ms_bvh_build"], "upload_ms": info["ms_upload"],
                         "build_threads": rt.build_threads, "triangles": info["n_triangles"], "bvh8_nodes": info["n_bvh_nodes"], "bvh8_depth": info["bvh_depth"],
                         "bytes_nodes": info["bytes_nodes"], "bytes_triangles": info["bytes_triangles"]},
               "roofline": roofline(workload, kt, n_node, n_tri, serial_ms)}
        if brief:
            res["protocol"] = (f"{steps} timed full step(s) ({full_spp} spp) after {warmup} warm-up step(s) at {short_spp} spp; per-kernel times from a "
                               f"{short_spp}-spp step scaled to {full_spp} spp (launch durations do not depend on the number of passes)")
        rt.close()
        return res

    line = dict(base_line)
    line.update(measure(args.workload, args.steps, max(args.warmup, 3), brief=False, dump_dir=args.dump_outputs))
    if also:
        line["also"] = {}
        for w in also:
            try:
                r = measure(w, 2 if w != "C5" else 1, 2, brief=True)
                r["workload"] = f"{w}: {WORKLOADS[w]}"
                line["also"][w] = r
            except Exception as e:      # a secondary workload never costs the main line
                line["also"][w] = {"workload": f"{w}: {WORKLOADS[w]}", "error": f"{type(e).__name__}: {e}"}
    if world > 1:
        dist.barrier()
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            try:
                cb, _, _ = cpu_reference(args.workload, 2, 1)
                line["cpu_baseline"] = cb
            except Exception as e:  # the baseline is a reported figure; never lose the GPU line over it
                line["cpu_baseline"] = {"value": None, "unit": "Msamples/s", "cores": None, "kind": "port", "sample": f"failed: {e}"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
