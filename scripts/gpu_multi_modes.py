"""The denoiser-input and progressive renderers on a group of N GPUs (ptb_group_*), N = 1, 2, 4, 8 as far as the box goes.
usage: python scripts/gpu_multi_modes.py TAG [OUT_DIR]   ->  OUT_DIR/TAG_multi_modes.jsonl (OUT_DIR defaults to profiles/)

  * denoiser inputs of C2 at 1024x1024, 64 spp, and the nopreviz render of the same scene: Msamples/s (best of 3, host outputs)
    and the ratio to N x one GPU;
  * the progressive renderer on C2 at 1920x1080: wall time of pass(passes_per_call) + read, for passes_per_call 1 and 16 (median of
    the calls; the read is where the gather is paid, so pass and read are also given apart)."""
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import pathtracer_b200 as ptb
from pathtracer_b200 import _abi, scenes

G = ptb.load()
TAG = sys.argv[1] if len(sys.argv) > 1 else "local"
OUT = os.path.join(sys.argv[2] if len(sys.argv) > 2 else os.path.join(ROOT, "profiles"), f"{TAG}_multi_modes.jsonl")
n_all = torch.cuda.device_count()
if n_all < 1:
    raise SystemExit("no CUDA device: this script measures the GPUs")
try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.splitlines()
except OSError:
    smi = []
BOX = {"gpu": smi[0].split(",")[0].strip() if smi else torch.cuda.get_device_name(0), "power_limit": smi[0].split(",")[1].strip() if smi else "unknown",
       "gpus_on_box": n_all}


def emit(rec):
    rec = {"tag": TAG, **BOX, **rec}
    print(json.dumps(rec), flush=True)
    with open(OUT, "a") as f:
        f.write(json.dumps(rec) + "\n")


def make(W, H, spp, n):
    rt = scenes.config_C2(G, W, H, spp)
    rt.devices = list(range(n)) if n > 1 else None
    return rt.commit()


def best_of(fn, reps=3):
    fn()                                  # warm-up: buffers, pools, the first launches
    best = 1e30
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); best = min(best, time.perf_counter() - t0)
    return best


def progressive(rt, ppc, calls):
    """median ms of pass(ppc), of read, and of the two together, over `calls` rounds of one session"""
    L, cam, p = G, rt.cam.c_struct(), rt.params()
    g, ctx = rt._group, rt._ctx
    n = C.c_int32(0)
    img, cnt = np.empty((rt.H, rt.W, 3), np.float32), np.empty((rt.H, rt.W), np.float32)
    u8, lr = np.empty((rt.H, rt.W, 3), np.uint8), np.empty((-(-rt.H // 16), -(-rt.W // 16), 3), np.float32)
    outs = (_abi.fptr(img), _abi.fptr(cnt), u8.ctypes.data_as(C.POINTER(C.c_uint8)), _abi.fptr(lr), C.byref(n))
    if g is not None:
        begin, step, read = (lambda: L.group_progressive_begin(g, C.byref(cam), C.byref(p)), lambda: L.group_progressive_pass(g, ppc, None),
                             lambda: L.group_progressive_read(g, *outs))
    else:
        begin, step, read = (lambda: L.progressive_begin(ctx, C.byref(cam), C.byref(p)), lambda: L.progressive_pass(ctx, ppc, None),
                             lambda: L.progressive_read(ctx, *outs))
    assert begin() == 0
    assert step() == 0 and read() == 0        # warm-up
    t_pass, t_read = [], []
    for _ in range(calls):
        t0 = time.perf_counter(); assert step() == 0
        t1 = time.perf_counter(); assert read() == 0
        t2 = time.perf_counter()
        t_pass.append((t1 - t0) * 1e3); t_read.append((t2 - t1) * 1e3)
    return statistics.median(t_pass), statistics.median(t_read), statistics.median(a + b for a, b in zip(t_pass, t_read)), float(img.sum() / max(float(cnt.sum()), 1.0))


one = {}
for n in [k for k in (1, 2, 4, 8) if k <= n_all]:
    rt = make(1024, 1024, 64, n)
    for mode, fn in (("denoiser_inputs", rt.render_denoiser_inputs), ("nopreviz", rt.render_image_nopreviz)):
        t = best_of(fn)
        msps = 1024 * 1024 * 64 / t / 1e6
        if n == 1:
            one[mode] = msps
        emit({"mode": mode, "scene": "C2", "W": 1024, "H": 1024, "spp": 64, "gpus": n, "ms_wall": round(t * 1e3, 3), "msamples_s": round(msps, 1),
              "ratio_to_n_x_1": round(msps / (n * one[mode]), 3), "samples": rt.stats["samples"], "mean": round(float(rt.imagedouble.mean()), 4)})
    rt.close()
    rt = make(1920, 1080, 1 << 20, n)
    for ppc, calls in ((1, 30), (16, 10)):
        tp, tr, tt, mean = progressive(rt, ppc, calls)
        emit({"mode": "progressive", "scene": "C2", "W": 1920, "H": 1080, "passes_per_call": ppc, "gpus": n, "calls": calls, "ms_pass": round(tp, 3),
              "ms_read": round(tr, 3), "ms_pass_plus_read": round(tt, 3), "msamples_s_pass_plus_read": round(1920 * 1080 * ppc / tt / 1e3, 1), "mean": round(mean, 4)})
    rt.close()
