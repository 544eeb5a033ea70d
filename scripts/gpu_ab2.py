"""One process = one library configuration (a variant library built with `make variant` is selected with PTB_LIB_PATH):
device ms per render for C2/C3/C4 at 1 and 2 pass pipelines, kernel breakdown and traversal counters.
usage: [ENV=...] python scripts/gpu_ab2.py <tag> [C2:256 C3:128 C4:256]"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pathtracer_b200 as ptb
from pathtracer_b200 import scenes, _abi

G = ptb.load()
tag = sys.argv[1]
specs = [a for a in sys.argv[2:] if ":" in a] or ["C2:256", "C3:128", "C4:256"]
for spec in specs:
    wl, spp = spec.split(":")
    rt = scenes.CONFIGS[wl](G); rt.nrays = int(spp); rt.commit()
    info = rt.scene_info()
    rt.set_option(_abi.OPT_COUNT_TRAVERSAL, 1); full = rt.nrays; rt.nrays = 4
    rt.render_image_nopreviz(want_image=False)
    kt = rt.kernel_times(); rt.nrays = full; rt.set_option(_abi.OPT_COUNT_TRAVERSAL, 0)
    n_node = kt["extend"]["node_visits"] / max(1, kt["extend"]["items"]); n_tri = kt["extend"]["tri_tests"] / max(1, kt["extend"]["items"])
    print(f"[{tag}] {wl}: nodes={info['n_bvh_nodes']} depth={info['bvh_depth']} build_ms={info['ms_bvh_build']:.0f} closest: n_node={n_node:.2f} n_tri={n_tri:.2f}", flush=True)
    for pipes, tb in ((1, int(os.environ.get("PTB_AB_TB", 9))), (2, 6)):
        rt.set_option(_abi.OPT_PIPES, pipes)
        rt.set_option(_abi.OPT_TRACE_BLOCKS, 148 * tb)
        best = 1e30
        for rep in range(3):
            img = rt.render_image_nopreviz(want_image=False)
            best = min(best, rt.stats["ms_device"])
        samples = rt.W * rt.H * rt.nrays
        line = f"[{tag}] {wl} spp={spp} pipes={pipes}: {best:9.2f} ms  {samples / best / 1e3:8.1f} Msamples/s mean={float(img.mean()):.4f}"
        if pipes == 1:
            rt.set_option(_abi.OPT_TIME_KERNELS, 1)
            rt.render_image_nopreviz(want_image=False)
            k = rt.kernel_times(); rt.set_option(_abi.OPT_TIME_KERNELS, 0)
            line += "  kernels ms: " + " ".join(f"{n}={v['ms']:.1f}" for n, v in k.items())
        print(line, flush=True)
    rt.close()
