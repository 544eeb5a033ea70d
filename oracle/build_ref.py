#!/usr/bin/env python3
"""Build oracle/_ref/libptb_ref.so: the REFERENCE's own renderer core, compiled headless.

TEST INFRASTRUCTURE ONLY.  Nothing in the product (pathtracer_b200/) may import, link or execute
anything produced here; only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs do.

The reference (the checkout of nbonneel/pathtracer given as the argument, read-only; tests/oracles.py passes the one
PTB_REFERENCE_DIR names) does not compile with GCC as shipped, so its sources are copied to a throw-away temp dir, patched there, compiled together with oracle/ref_driver.cpp (ours)
and the temp dir is deleted.  No reference source enters the repo; the only output is the .so under
oracle/_ref/ (git-ignored, travels to the GPU box).

Patches applied to the temp copy (each must match exactly once, else the build aborts):
  1. Vector.h      random_uniform_sphere() inside a template needs <T>            (compile fix)
  2. Raytracer.cpp `Vector& axis = -N;` binds a non-const ref to a temporary      (compile fix)
  3. Raytracer.cpp unbalanced braces when USE_OPENIMAGEDENOISER is undefined      (compile fix)
  4. Vector.h      invSqRoot reads a float through long* (8 bytes on LP64)        (correctness on Linux:
                   the author's Windows build has 4-byte long; int32_t restores the intended behaviour)
  5. Raytracer.cpp per-(pixel,sample) pcg32 streams instead of per-thread engines (determinism; this
                   is the inline ray generation the author left commented at Raytracer.cpp:1613-1622,
                   preceded by a reseed; see DESIGN.md "RNG"); 5c: the same reseed in front of the
                   draws of the progressive renderer render_image (Raytracer.cpp:1462)
  6. Geometry.cpp  per-thread ray counters at the top of Scene::intersection{,_shadow} (measurement)
  7. Raytracer.h/.cpp  every `Contrib` of getColor's ring carries its own pcg32 (determinism under branching:
                   fog and ghost objects push more than one contribution per iteration, and the ring interleaves
                   their draws).  The continuation of a path keeps the path's stream, so non-branching renders draw
                   exactly what patch 5 alone gives; a side branch (the in-scattering contribution of
                   fogContribution, the straight-through ray of a ghost object) starts
                   ptb_fork(engine, tag) = pcg32(seed = two draws of a COPY of the parent engine, stream = tag),
                   tag 1 = fog, 2 = ghost.  `float attenuationFactor;` (read uninitialised when the first
                   fogContribution of a sample returns early) starts at 1.
Flags: -std=c++11 -O2 -fopenmp -fpermissive -include omp.h -D__forceinline=inline, unity TU.
"""
import os
import re
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")

UNITY = ["Vector.cpp", "Geometry.cpp", "TriangleMesh.cpp", "PointSet.cpp", "fluid.cpp", "Raytracer.cpp"]
SEPARATE = ["MERLBRDFRead.cpp", "utils.cpp", "hdrwriter.cpp", "hdrloader.cpp"]


def sub_once(text, pattern, repl, what, flags=0):
    new, n = re.subn(pattern, repl, text, flags=flags)
    if n != 1:
        raise SystemExit(f"build_ref: patch '{what}' matched {n} times (expected 1)")
    return new


def patch(tmp):
    def rd(name):
        with open(os.path.join(tmp, name), "r", encoding="latin-1", newline="") as f:
            return f.read()

    def wr(name, text):
        with open(os.path.join(tmp, name), "w", encoding="latin-1", newline="") as f:
            f.write(text)

    v = rd("Vector.h")
    v = sub_once(v, r"T\(1\. / 3\.\)\)\*random_uniform_sphere\(\);",
                 "T(1. / 3.))*random_uniform_sphere<T>();", "1 random_uniform_sphere<T>")
    v = sub_once(v, r"long i = \*\(long \*\)&y;", "int32_t i = *(int32_t *)&y;", "4 invSqRoot pun")
    wr("Vector.h", v)

    h = rd("Raytracer.h")
    h = sub_once(h, r"(bool show_lights, has_had_subsurface_interaction, showenvmap;\s*\n)(\};)",
                 r"\1\tpcg32 ptb_rng;\n\2\n"
                 r"static inline pcg32 ptb_fork(const pcg32& e, uint64_t tag) { pcg32 t = e; uint64_t a = t(); uint64_t b = t(); return pcg32((a << 32) | b, tag); }\n",
                 "7a Contrib rng")
    wr("Raytracer.h", h)

    r = rd("Raytracer.cpp")
    r = sub_once(r, r"Vector& axis = -N;", "Vector axis = -N;", "2 axis ref")
    # 3: close the `else {` of the has_denoiser branch when OIDN is absent: the LAST #endif of the file
    idx = r.rfind("#endif")
    if idx < 0:
        raise SystemExit("build_ref: patch 3: no #endif")
    r = r[:idx] + "#else\n\t}\n#endif" + r[idx + len("#endif"):]
    # 5: per-(pixel,sample) RNG
    r = sub_once(r, r"\n[ \t]*precomputeRayBatch\(batchi\*batchHeight,[^\n]*nrays\);", "\n", "5a drop precompute")
    r = sub_once(
        r,
        r"const Ray &r = s\.firstIntersection_Ray\[threadid\]\[id\*nrays\+k\];\s*"
        r"float dx = s\.firstIntersection_dx\[threadid\]\[id\*nrays \+ k\];\s*"
        r"float dy = s\.firstIntersection_dy\[threadid\]\[id\*nrays \+ k\];\s*"
        r"Vector normal, albedo;\s*"
        r"Vector color = getColor\(r, k, nb_bounces, i, j, normal, albedo, false, true, id\*nrays \+ k\);",
        "engine[threadid] = pcg32((uint64_t)(i*W + j), (uint64_t)k ^ ((uint64_t)ptb_ref_global_seed << 32));\n"
        "float dx = engine[threadid]()*invmax - 0.5f;\n"
        "float dy = engine[threadid]()*invmax - 0.5f;\n"
        "float dx_aperture = (engine[threadid]()*invmax - 0.5f) * cam.aperture;\n"
        "float dy_aperture = (engine[threadid]()*invmax - 0.5f) * cam.aperture;\n"
        "float time = s.current_frame;\n"
        "Ray r = cam.generateDirection(s.double_frustum_start_t, i, j, time, dx, dy, dx_aperture, dy_aperture, W, H);\n"
        "Vector normal, albedo;\n"
        "Vector color = getColor(r, k, nb_bounces, i, j, normal, albedo, false, false);",
        "5b inline per-sample rays")
    # 5c: the same per-(pixel,sample) stream in the progressive renderer (render_image, Raytracer.cpp:1459-1466)
    r = sub_once(
        r,
        r"(for \(int j = j1; j < W; j \+= 8\) \{\s*)(float dx = engine\[threadid\]\(\)\*invmax - 0\.5f;)",
        r"\1engine[threadid] = pcg32((uint64_t)(i*W + j), (uint64_t)realtime_ray_iter ^ ((uint64_t)ptb_ref_global_seed << 32));\n\2",
        "5c progressive per-sample streams")
    # 7: per-contribution engines, inside the live getColor only (a second copy sits under `#if 0`)
    g0 = r.index("Vector Raytracer::getColor(")
    g1 = r.index("#if 0", g0)
    body = r[g0:g1]

    def sub_n(text, pattern, repl, n_expected, what):
        new, n = re.subn(pattern, repl, text)
        if n != n_expected:
            raise SystemExit(f"build_ref: patch '{what}' matched {n} times (expected {n_expected})")
        return new
    body = sub_n(body, r"float attenuationFactor;", "float attenuationFactor = 1.f;", 1, "7b attenuationFactor")
    body = sub_n(body, r"(contribs\[contribIndexStart\] = Contrib\(Vector\(1\.f, 1\.f, 1\.f\), r, nb_bounces, true, false\);)",
                 r"\1 contribs[contribIndexStart].ptb_rng = engine[threadid];", 1, "7c root engine")
    body = sub_n(body, r"(const Contrib& curContrib = contribs\[contribIndexStart\];)", r"\1 engine[threadid] = curContrib.ptb_rng;", 1, "7d pop engine")
    body = sub_n(body, r"(contribs\[contribIndexEnd\] = newContrib;)", r"\1 contribs[contribIndexEnd].ptb_rng = ptb_fork(engine[threadid], 1);", 6, "7e fog fork")
    body = sub_n(body, r"(contribs\[contribIndexEnd\] = Contrib\(pathWeight, currentRay, nbrebonds, show_lights, has_had_subsurface_interaction, show_envmap\);)",
                 r"\1 contribs[contribIndexEnd].ptb_rng = ptb_fork(engine[threadid], 2);", 1, "7f ghost fork")
    body = sub_n(body, r"(contribs\[contribIndexEnd\] = Contrib\((?:attenuationFactor\*)?(?:pathWeight|newpathWeight), (?:rayon_miroir|new_ray|rayon_aleatoire),[^\n]*\);)",
                 r"\1 contribs[contribIndexEnd].ptb_rng = engine[threadid];", 6, "7g continuation engine")
    r = r[:g0] + body + r[g1:]
    wr("Raytracer.cpp", r)

    g = rd("Geometry.cpp")
    g = sub_once(
        g,
        r"(bool Scene::intersection\(const Ray& d, Vector& P, int &sphere_id, float &min_t, MaterialValues &mat, int &triangle_id, bool avoid_ghosts, bool isCoherent\) const \{)",
        r"\1\n\tptb_ref_cnt[omp_get_thread_num()][0]++;", "6a closest counter")
    g = sub_once(
        g,
        r"(bool Scene::intersection_shadow\(const Ray& d, float &min_t, float dist_light, bool avoid_ghosts, bool isCoherent\) const \{)",
        r"\1\n\tptb_ref_cnt[omp_get_thread_num()][1]++;", "6b shadow counter")
    wr("Geometry.cpp", g)


def main(argv):
    if len(argv) != 2 or not os.path.isdir(argv[1]):
        print("usage: build_ref.py <checkout of nbonneel/pathtracer>", file=sys.stderr)
        return 2
    REF = argv[1]
    os.makedirs(OUT, exist_ok=True)
    tmp = tempfile.mkdtemp(prefix="ptb_ref_build_")
    try:
        for name in os.listdir(REF):
            if name.startswith("mainApp"):
                continue
            if name.endswith((".cpp", ".h", ".hpp")):
                shutil.copy(os.path.join(REF, name), os.path.join(tmp, name))
        patch(tmp)
        cxx = os.environ.get("PTB_CXX", "g++")  # NB: $CXX in this image points at a g++ without libgomp.spec
        flags = ["-std=c++11", "-O2", "-fopenmp", "-fpermissive", "-w", "-fPIC",
                 "-include", "omp.h", "-D__forceinline=inline", f"-I{tmp}",
                 f"-I{os.path.join(HERE, '..', 'include')}", f"-I{HERE}"]
        objs = []
        for src in SEPARATE:
            obj = os.path.join(tmp, src[:-4] + ".o")
            subprocess.check_call([cxx, *flags, "-c", os.path.join(tmp, src), "-o", obj])
            objs.append(obj)
        unity = os.path.join(tmp, "unity.cpp")
        with open(unity, "w") as f:
            f.write('#include <stdint.h>\n#include <omp.h>\n')
            f.write('extern uint32_t ptb_ref_global_seed;\nextern unsigned long long ptb_ref_cnt[64][8];\n')
            f.write('#include "chrono.h"\n')
            for src in UNITY:
                f.write(f'#include "{src}"\n')
            f.write(f'#include "{os.path.join(HERE, "ref_driver.cpp")}"\n')
        so = os.path.join(OUT, "libptb_ref.so")
        subprocess.check_call([cxx, *flags, "-shared", unity, *objs, "-o", so])
        print(f"build_ref: wrote {so}")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv))
