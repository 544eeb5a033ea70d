// ptb_core.h — POD types and the small numeric building blocks of the radiance loop.
//
// Everything here is written once as `PTB_HD` inline functions.  nvcc compiles them for sm_100a as
// the bodies of the CUDA kernels in kernels.cu (the product).  tests/devsim compiles the same
// headers with g++ to step the device logic on the CPU while debugging without a GPU; that build is
// test-only and is not part of libptb200.so (tests/test_abi.py checks the library has no such symbols).
//
// Numerics follow the reference's float32 arithmetic operation by operation where the reference
// computes in float, and keep its double intermediates where they change the rounded result
// (fast_exp, extensibleLattice2d, the MERL lookup).  Citations are into /root/reference.
#pragma once
#include <stdint.h>
#include <math.h>
#include <string.h>

#if defined(__CUDACC__)
#define PTB_HD __host__ __device__ __forceinline__
#define PTB_D __device__ __forceinline__
#else
#define PTB_HD inline
#define PTB_D inline
#endif
#if defined(__CUDA_ARCH__)
#define PTB_HD_NOINLINE __host__ __device__ __noinline__
#elif defined(__CUDACC__)
#define PTB_HD_NOINLINE __host__ __device__
#else
#define PTB_HD_NOINLINE inline
#endif

#define PTB_PI_F 3.14159274101257324f            /* float(M_PI) */
#define PTB_PI_D 3.1415926535897932              /* M_PI as the reference defines it, Vector.h:8-10 */
#define PTB_TWO_PI_REF 6.28318530718             /* M_TWO_PI, Vector.h:16-18 (NOT 2*M_PI to the last bit) */

namespace ptb {

struct V3 {
    float x, y, z;
};
struct alignas(16) F4 {
    float x, y, z, w;
};
struct alignas(16) U4 {
    uint32_t x, y, z, w;
};
struct alignas(8) U2 {
    uint32_t x, y;
};

PTB_HD V3 v3(float x, float y, float z) { V3 r; r.x = x; r.y = y; r.z = z; return r; }
PTB_HD V3 operator+(V3 a, V3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
PTB_HD V3 operator-(V3 a, V3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
PTB_HD V3 operator-(V3 a) { return v3(-a.x, -a.y, -a.z); }
PTB_HD V3 operator*(V3 a, V3 b) { return v3(a.x * b.x, a.y * b.y, a.z * b.z); }
PTB_HD V3 operator*(float s, V3 a) { return v3(s * a.x, s * a.y, s * a.z); }
PTB_HD V3 operator*(V3 a, float s) { return v3(s * a.x, s * a.y, s * a.z); }
PTB_HD V3 operator/(V3 a, float s) { return v3(a.x / s, a.y / s, a.z / s); }
// dot() as the reference writes it (Vector.h:553-556): a0*b0 + a1*b1 + a2*b2, left to right.
// __fmaf_rn contraction is left to the compiler (nvcc -fmad=true): see DESIGN.md "rounding".
PTB_HD float dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
PTB_HD float norm2(V3 a) { return a.x * a.x + a.y * a.y + a.z * a.z; }
PTB_HD V3 cross(V3 a, V3 b) { return v3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
// VectorT::normalize (Vector.h:371-376): divide by sqrt(norm2)
PTB_HD V3 normalize(V3 a) {
    float n = sqrtf(norm2(a));
    return v3(a.x / n, a.y / n, a.z / n);
}
// VectorT::reflect (Vector.h:388-391): d - 2 (d.N) N
PTB_HD V3 reflect(V3 d, V3 N) { return d - (2.f * dot(d, N)) * N; }

// ---- the reference's float arithmetic, operation by operation ---------------------------------------------------------------------
// nvcc contracts a*b+c into one FMA (one rounding), the reference's x86-64 build rounds twice.  Where a DECISION of the reference has
// to be reproduced and not just its value (which triangle a ray near a shared edge hits, which texel an alpha lookup reads), the
// operations are spelled with the round-to-nearest intrinsics, which are never contracted, in the reference's order.  (The host
// compilations of these headers, tests/devsim, use -ffp-contract=off.)
#if defined(__CUDA_ARCH__)
PTB_HD float mul_rn(float a, float b) { return __fmul_rn(a, b); }
PTB_HD float add_rn(float a, float b) { return __fadd_rn(a, b); }
PTB_HD float sub_rn(float a, float b) { return __fsub_rn(a, b); }
PTB_HD float div_rn(float a, float b) { return __fdiv_rn(a, b); }
PTB_HD float sqrt_rn(float a) { return __fsqrt_rn(a); }
#else
PTB_HD float mul_rn(float a, float b) { return a * b; }
PTB_HD float add_rn(float a, float b) { return a + b; }
PTB_HD float sub_rn(float a, float b) { return a - b; }
PTB_HD float div_rn(float a, float b) { return a / b; }
PTB_HD float sqrt_rn(float a) { return sqrtf(a); }
#endif
PTB_HD float dot_rn(V3 a, V3 b) { return add_rn(add_rn(mul_rn(a.x, b.x), mul_rn(a.y, b.y)), mul_rn(a.z, b.z)); }     // Vector.h:553-556
PTB_HD V3 cross_rn(V3 a, V3 b) {
    return v3(sub_rn(mul_rn(a.y, b.z), mul_rn(a.z, b.y)), sub_rn(mul_rn(a.z, b.x), mul_rn(a.x, b.z)), sub_rn(mul_rn(a.x, b.y), mul_rn(a.y, b.x)));
}
PTB_HD V3 add3_rn(V3 a, V3 b) { return v3(add_rn(a.x, b.x), add_rn(a.y, b.y), add_rn(a.z, b.z)); }
PTB_HD V3 sub3_rn(V3 a, V3 b) { return v3(sub_rn(a.x, b.x), sub_rn(a.y, b.y), sub_rn(a.z, b.z)); }
PTB_HD V3 scale_rn(float s, V3 a) { return v3(mul_rn(s, a.x), mul_rn(s, a.y), mul_rn(s, a.z)); }
PTB_HD V3 normalize_rn(V3 a) {                                                                                       // Vector.h:371-376
    const float n = sqrt_rn(dot_rn(a, a));
    return v3(div_rn(a.x, n), div_rn(a.y, n), div_rn(a.z, n));
}

PTB_HD uint32_t f2u(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
PTB_HD float u2f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }

// invSqRoot (Vector.h:294-309) with the 32-bit pun the author's platform has: magic constant,
// two Newton steps.  fast_normalize (Vector.h:376-382) multiplies by it.
PTB_HD float inv_sq_root(float n) {
    float y = n;
    int32_t i = (int32_t)f2u(y);
    i = 0x5f3759df - (i >> 1);
    y = u2f((uint32_t)i);
    y = y * (1.5f - ((n * 0.5f) * y * y));
    y = y * (1.5f - ((n * 0.5f) * y * y));
    return y;
}
PTB_HD V3 fast_normalize(V3 a) {
    float inv = inv_sq_root(norm2(a));
    return v3(a.x * inv, a.y * inv, a.z * inv);
}

// ---- pcg32 = setseq_xsh_rr_64_32 (pcg_random.hpp:1866, 845-873, 484-501, 158-159) ----------------
#define PTB_PCG_MULT 6364136223846793005ULL
#define PTB_PCG_DEFAULT_INC 1442695040888963407ULL
struct Pcg32 {
    uint64_t state, inc;
};
PTB_HD Pcg32 pcg32_seed(uint64_t state_seed, uint64_t stream) {  // two-argument ctor, pcg_random.hpp:494-501
    Pcg32 r;
    r.inc = (stream << 1) | 1ULL;
    r.state = (state_seed + r.inc) * PTB_PCG_MULT + r.inc;
    return r;
}
PTB_HD uint32_t pcg32_next(Pcg32& r) {  // output function applied to the PRE-advance state
    uint64_t old = r.state;
    r.state = old * PTB_PCG_MULT + r.inc;
    uint32_t xorshifted = (uint32_t)(((old >> 18u) ^ old) >> 27u);
    uint32_t rot = (uint32_t)(old >> 59u);
    return (xorshifted >> rot) | (xorshifted << ((32u - rot) & 31u));
}
// engine()*invmax with invmax = 1.f/engine.max() = 2^-32 (Raytracer.h:28): closed [0,1]
PTB_HD float pcg32_uniform(Pcg32& r) { return (float)pcg32_next(r) * 2.3283064365386963e-10f; }
// per-(pixel,sample) stream, DESIGN.md "RNG" (SURVEY App. C)
PTB_HD Pcg32 pcg32_for_sample(uint32_t pixel, uint32_t k, uint32_t seed) {
    return pcg32_seed((uint64_t)pixel, (uint64_t)k ^ ((uint64_t)seed << 32));
}
// LCG jump-ahead (pcg_random.hpp `advance`): state after `delta` steps
PTB_HD uint64_t pcg_advance(uint64_t state, uint64_t delta, uint64_t mult, uint64_t inc) {
    uint64_t acc_mult = 1, acc_plus = 0;
    while (delta > 0) {
        if (delta & 1) {
            acc_mult *= mult;
            acc_plus = acc_plus * mult + inc;
        }
        inc = (mult + 1) * inc;
        mult *= mult;
        delta >>= 1;
    }
    return acc_mult * state + acc_plus;
}
// randomPerPixel[p] = draws 2p and 2p+1 of pcg32(0) (Raytracer.cpp:1325-1345)
PTB_HD void random_per_pixel(uint32_t p, float& rx, float& ry) {
    Pcg32 e;
    e.inc = PTB_PCG_DEFAULT_INC;
    e.state = (0ULL + e.inc) * PTB_PCG_MULT + e.inc;
    e.state = pcg_advance(e.state, 2ULL * p, PTB_PCG_MULT, e.inc);
    rx = pcg32_uniform(e);
    ry = pcg32_uniform(e);
}

// ---- extensibleLattice2d (Raytracer.cpp:1302-1319) ------------------------------------------------
PTB_HD uint32_t reverse_bits(uint32_t n) {
#if defined(__CUDA_ARCH__)
    return __brev(n);
#else
    n = (n << 16) | (n >> 16);
    n = ((n & 0x00ff00ffu) << 8) | ((n & 0xff00ff00u) >> 8);
    n = ((n & 0x0f0f0f0fu) << 4) | ((n & 0xf0f0f0f0u) >> 4);
    n = ((n & 0x33333333u) << 2) | ((n & 0xccccccccu) >> 2);
    n = ((n & 0x55555555u) << 1) | ((n & 0xaaaaaaaau) >> 1);
    return n;
#endif
}
PTB_HD float frac_pos(float x) { return x - truncf(x); }  // modf(float,&ip) fractional part
PTB_HD void extensible_lattice_2d(uint32_t id, float& x, float& y) {
    uint32_t rid = reverse_bits(id);
    float phi = (float)((double)rid * 2.3283064365386963e-10);  // rid * pow(2.0,-32), narrowed to float
    // the sums are evaluated in double, narrowed to float by the modf(float,float*) overload, then reduced
    x = frac_pos((float)((double)(phi * 1.f) + 0.456789123));
    y = frac_pos((float)((double)(phi * 182667.f) + 0.123456789));
}

// ---- fast_exp (Raytracer.cpp:1294-1299), Schraudolph ----------------------------------------------
PTB_HD double fast_exp(double y) {
    int32_t hi = (int32_t)(1512775 * y + 1072632447);
    uint64_t bits = ((uint64_t)(uint32_t)hi) << 32;
    double d;
    memcpy(&d, &bits, 8);
    return d;
}

// x^y, x >= 0, as the device affords it: exp2f(y * log2f(x)), each accurate to an ulp, so the result is off the correctly rounded power by
// about |y log2 x| * 6e-8 relative (Ne = 100 at d = 0.9: 1e-6, far inside the 1e-4 of the phong_eval KAT), in 40 instructions where
// powf takes 96 (ncu r02t: the powf calls were 13 % of k_shade's instructions).  0^0 = 1 like powf; a negative x gives NaN where powf
// has a value for integer y: both callers discard the sample then (phong_eval returns before, phong_sample's caller tests dot(R, dir) < 0).
#if defined(__CUDA_ARCH__)
__device__ __forceinline__ float pow_pos(float x, float y) { const float r = exp2f(y * log2f(x)); return y == 0.f ? 1.f : r; }
#else
inline float pow_pos(float x, float y) { return powf(x, y); }
#endif
PTB_HD float pow5(float x) {      // Schlick's (1 - cos)^5 (Raytracer.cpp:459-462: std::pow(x, 5.f))
#if defined(__CUDA_ARCH__)
    const float x2 = x * x;
    return x2 * x2 * x;
#else
    return powf(x, 5.f);
#endif
}

// ---- getTangent / random_cos (Vector.h:566-600), random_Phong (BRDF.h:41-61) -----------------------
PTB_HD V3 get_tangent(V3 N) {
    float ax = fabsf(N.x), ay = fabsf(N.y), az = fabsf(N.z);
    V3 t;
    if (ax <= ay && ax <= az) t = v3(0.f, -N.z, N.y);
    else if (ay <= ax && ay <= az) t = v3(-N.z, 0.f, N.x);
    else t = v3(-N.y, N.x, 0.f);
    return normalize(t);
}
PTB_HD V3 random_cos(V3 N, float r1, float r2) {
    float sr2 = sqrtf(1.f - r2);
    float a = PTB_PI_F * 2.f * r1;  // T(2.*M_PI)*r1 : float(2pi) == 2*float(pi) exactly
#if defined(__CUDA_ARCH__)
    // one shared argument reduction instead of two (measured r01k: k_shade -3.5 % on C2, -2.3 % on C4; out-of-lining random_cos /
    // phong_eval to shrink the 84 KB kernel was measured too and is SLOWER by 2 %)
    // (r02u: sincospif of 2 r1: no Payne-Hanek path, a third of the instructions; the angle is not rounded to float first, which moves
    // the direction by at most 4e-7, inside the KAT's 2e-6)
    float sn, cs;
    sincospif(2.f * r1, &sn, &cs);
    float lx = cs * sr2, ly = sn * sr2, lz = sqrtf(r2);
#else
    float lx = cosf(a) * sr2, ly = sinf(a) * sr2, lz = sqrtf(r2);
#endif
    V3 t1 = get_tangent(N);
    V3 t2 = cross(t1, N);
    return lz * N + lx * t1 + ly * t2;
}
PTB_HD V3 random_phong(V3 R, float n, float r1, float r2) {
    float facteur = sqrtf(1.f - pow_pos(r2, 2.f / (n + 1.f)));
#if defined(__CUDA_ARCH__)
    // The reference evaluates cos/sin(2*pi*r1) and r2^(1/(n+1)) in double and narrows (BRDF.h:44).  On the device the
    // float functions are used: the results agree to 2 ulp (KAT tolerance 2e-5) and the double versions cost ~500
    // instructions for the fifth of the lanes that take the specular lobe.
    float sn, cs;
    sincospif(2.f * r1, &sn, &cs);
    float lx = cs * facteur, ly = sn * facteur, lz = pow_pos(r2, 1.f / (n + 1.f));
#else
    double a = 2 * PTB_PI_D * (double)r1;
    float lx = (float)(cos(a) * (double)facteur);
    float ly = (float)(sin(a) * (double)facteur);
    float lz = (float)pow((double)r2, 1. / (double)(n + 1.f));
#endif
    V3 t1 = get_tangent(R);
    V3 t2 = cross(t1, R);
    return lz * R + lx * t1 + ly * t2;
}

// ---- PhongBRDF (BRDF.h:63-96) ---------------------------------------------------------------------
PTB_HD V3 phong_eval(V3 Kd, V3 Ks, V3 Ne, V3 wi, V3 wo, V3 N) {
    V3 refl = reflect(-wo, N);
    float d = dot(refl, wi);
    V3 diff = Kd / PTB_PI_F;
    if (d < 0) return diff;
    V3 lobe;
#if defined(__CUDA_ARCH__)
    // float division by float(M_TWO_PI): within 1 ulp of the reference's double division + narrowing
    const float two_pi = (float)PTB_TWO_PI_REF;
    const bool same = (Ne.x == Ne.y) && (Ne.y == Ne.z);
    lobe.x = pow_pos(d, Ne.x) * (Ne.x + 2.f) / two_pi;
    lobe.y = same ? lobe.x : pow_pos(d, Ne.y) * (Ne.y + 2.f) / two_pi;
    lobe.z = same ? lobe.x : pow_pos(d, Ne.z) * (Ne.z + 2.f) / two_pi;
#else
    lobe.x = (float)((double)(powf(d, Ne.x) * (Ne.x + 2.f)) / PTB_TWO_PI_REF);
    lobe.y = (float)((double)(powf(d, Ne.y) * (Ne.y + 2.f)) / PTB_TWO_PI_REF);
    lobe.z = (float)((double)(powf(d, Ne.z) * (Ne.z + 2.f)) / PTB_TWO_PI_REF);
#endif
    return diff + lobe * Ks;
}
// sample(): `u` is the one extra engine draw (BRDF.h:73); returns direction, pdf, sampled-diffuse flag
PTB_HD V3 phong_sample(V3 Ks, V3 Ne, V3 wo, V3 N, float r1, float r2, float u, float& pdf, bool& diffuse) {
    float avgNe = (Ne.x + Ne.y + Ne.z) / 3.f;
    float p = 1 - (Ks.x + Ks.y + Ks.z) / 3.f;
    V3 R = reflect(-wo, N);
    V3 dir;
    if (u < p) { diffuse = true; dir = random_cos(N, r1, r2); }
    else { diffuse = false; dir = random_phong(R, avgNe, r1, r2); }
#if defined(__CUDA_ARCH__)
    float proba_phong = (avgNe + 1) / (2.f * PTB_PI_F) * pow_pos(dot(R, dir), avgNe);
    pdf = (p * dot(N, dir)) / PTB_PI_F + (1.f - p) * proba_phong;
#else
    float proba_phong = (float)((double)(avgNe + 1) / (2.f * PTB_PI_D) * (double)powf(dot(R, dir), avgNe));
    pdf = (float)((double)(p * dot(N, dir)) / PTB_PI_D + (double)((1.f - p) * proba_phong));
#endif
    return dir;
}

// ---- IsoMERLBRDF (BRDF.h:204-246) + lookup_brdf_val (MERLBRDFRead.cpp:76-207), all in double -------
// `table` holds the three channels PRE-MULTIPLIED by their scale and narrowed to float exactly as
// `result[c] = (float)(brdf[ind + c*N] * SCALE_c)` does in the reference (BRDF.h:240-243).
PTB_HD void merl_rotate(const double* v, const double* axis, double angle, double* out) {
    double c = cos(angle), s = sin(angle);
    out[0] = v[0] * c; out[1] = v[1] * c; out[2] = v[2] * c;
    double temp = axis[0] * v[0] + axis[1] * v[1] + axis[2] * v[2];
    temp = temp * (1.0 - c);
    out[0] += axis[0] * temp; out[1] += axis[1] * temp; out[2] += axis[2] * temp;
    double cr[3] = {axis[1] * v[2] - axis[2] * v[1], axis[2] * v[0] - axis[0] * v[2], axis[0] * v[1] - axis[1] * v[0]};
    out[0] += cr[0] * s; out[1] += cr[1] * s; out[2] += cr[2] * s;
}
// Out of line on the device: it is the rare fallback of merl_index_fast, and inlined it dictates the register allocation of the
// whole shade kernel (102 registers, 5 blocks/SM).
PTB_HD_NOINLINE int merl_index(double theta_in, double fi_in, double theta_out, double fi_out) {
    const double MPI = 3.1415926535897932384626433832795;
    double in_z = cos(theta_in), pin = sin(theta_in);
    double in_x = pin * cos(fi_in), in_y = pin * sin(fi_in);
    double in[3] = {in_x, in_y, in_z};
    double len = sqrt(in[0] * in[0] + in[1] * in[1] + in[2] * in[2]);
    in[0] /= len; in[1] /= len; in[2] /= len;
    double out_z = cos(theta_out), pout = sin(theta_out);
    double out_x = pout * cos(fi_out), out_y = pout * sin(fi_out);
    // (the reference normalises `out` too but then uses the un-normalised components for the half vector)
    double h[3] = {(in_x + out_x) / 2.0, (in_y + out_y) / 2.0, (in_z + out_z) / 2.0};
    len = sqrt(h[0] * h[0] + h[1] * h[1] + h[2] * h[2]);
    h[0] /= len; h[1] /= len; h[2] /= len;
    double theta_half = acos(h[2]);
    double fi_half = atan2(h[1], h[0]);
    const double bi_normal[3] = {0.0, 1.0, 0.0}, normal[3] = {0.0, 0.0, 1.0};
    double temp[3], diff[3];
    merl_rotate(in, normal, -fi_half, temp);
    merl_rotate(temp, bi_normal, -theta_half, diff);
    double theta_diff = acos(diff[2]);
    double fi_diff = atan2(diff[1], diff[0]);
    // theta_half_index
    int ih;
    if (theta_half <= 0.0) ih = 0;
    else {
        double deg = ((theta_half / (MPI / 2.0)) * 90);
        double t = sqrt(deg * 90);
        ih = (int)t;
        if (ih < 0) ih = 0;
        if (ih >= 90) ih = 89;
    }
    // theta_diff_index
    int id = (int)(theta_diff / (MPI * 0.5) * 90);
    if (id < 0) id = 0; else if (id >= 89) id = 89;
    // phi_diff_index
    if (fi_diff < 0.0) fi_diff += MPI;
    int ip = (int)(fi_diff / MPI * 360 / 2);
    if (ip < 0) ip = 0; else if (ip >= 179) ip = 179;
    return ip + id * 180 + ih * 180 * 90;
}
#define PTB_MERL_N (90 * 90 * 180)
// Float evaluation of the same three bin positions with a guard band.  The double path above costs about a third of k_shade's
// instructions on the MERL configuration (12 double sin/cos, 2 acos, 2 atan2, 3 sqrt, 6 divisions per lookup), but its result is
// three small integers: the float path computes the CONTINUOUS bin positions from the local unit vectors (no angles: the Rodrigues
// rotations by -phi_h and -theta_h are written with cos/sin taken from the half vector), and answers only when every position is
// farther from a bin edge than a bound on everything that separates the two evaluations (the reference's float acosf/atan2f of
// the inputs, 1-3 ulp; float rounding here): 1.5e-6 on the unit vectors, propagated to each position.  Otherwise it returns false
// and the caller runs the double path, so the bin index is the reference's in both cases (checked against the double path on 1e8
// random direction pairs by tests/test_host_logic.py::test_merl_index_fast, and on the device by the MERL KAT).
#define PTB_MERL_EPS0 2.5e-6f   /* device atan2f: 2 ulp of an azimuth up to 2 pi = 1e-6; acosf; the float arithmetic here */
PTB_HD bool merl_index_fast(V3 wil, V3 wol, int& ind) {
    const float HALF_PI = 1.57079632679489662f, INV_PI_180 = 57.2957795130823209f;   // 180/pi = 90/(pi/2)
    // the reference goes through theta = acosf(z), phi = atan2f(y, x) and rebuilds (sin theta cos phi, sin theta sin phi, cos theta):
    // z is kept AS IS (the local vectors are only approximately unit: the shading normal comes from fast_normalize) and (x, y) only
    // give the azimuth
    const float ri2 = wil.x * wil.x + wil.y * wil.y, ro2 = wol.x * wol.x + wol.y * wol.y;
    if (!(ri2 > 1e-12f && ro2 > 1e-12f)) return false;
    const float si = sqrtf((1.f - wil.z) * (1.f + wil.z)) / sqrtf(ri2), so = sqrtf((1.f - wol.z) * (1.f + wol.z)) / sqrtf(ro2);
    const V3 in = v3(wil.x * si, wil.y * si, wil.z), out = v3(wol.x * so, wol.y * so, wol.z);
    V3 h = in + out;
    const float hl2 = dot(h, h);
    if (!(hl2 > 1e-4f)) return false;
    const float rhl = 1.f / sqrtf(hl2);
    h = h * rhl;
    const float sh2 = h.x * h.x + h.y * h.y;
    if (!(sh2 > 1e-6f)) return false;               // theta_half < 1e-3: phi_half (and with it phi_diff) is ill-conditioned
    const float sh = sqrtf(sh2), ch = h.z, rsh = 1.f / sh;
    const float cp = h.x * rsh, sp = h.y * rsh;
    const float tx = cp * in.x + sp * in.y, ty = cp * in.y - sp * in.x, tz = in.z;     // rotation by -phi_half about the normal
    const float dx = ch * tx - sh * tz, dy = ty, dz = sh * tx + ch * tz;               // rotation by -theta_half about the bi-normal
    const float sd2 = dx * dx + dy * dy;
    if (!(sd2 > 1e-6f)) return false;               // theta_diff < 1e-3: phi_diff is ill-conditioned
    const float sd = sqrtf(sd2);
    const float theta_half = atan2f(sh, ch), theta_diff = atan2f(sd, dz);
    float fi_diff = atan2f(dy, dx);
    if (fi_diff < 0.f) fi_diff += 3.14159265358979323846f;
    const float ph = sqrtf(theta_half * (8100.f / HALF_PI));   // sqrt(theta_half / (pi/2) * 90 * 90)
    const float pd = theta_diff * INV_PI_180;
    const float pp = fi_diff * INV_PI_180;
    // error propagation: each unit vector is uncertain by EPS0 plus what the reference loses by going through theta = acosf(z)
    // (z is quantised to 6e-8 next to 1: 1.2e-7 / sin theta) -> the half vector (cancellation in in + out: / |in + out|) ->
    // theta_half, and phi_half (/ sin theta_half) -> the rotated vector -> theta_diff, and phi_diff (/ sin theta_diff); then
    // d(position)/d(angle)
    const float si2 = in.x * in.x + in.y * in.y, so2 = out.x * out.x + out.y * out.y;
    if (!(si2 > 1e-8f && so2 > 1e-8f)) return false;
    const float ei = PTB_MERL_EPS0 + 1.2e-7f / sqrtf(si2), eo = PTB_MERL_EPS0 + 1.2e-7f / sqrtf(so2);
    const float eh = (ei + eo) * rhl;
    const float ed = ei + eh * (1.f + rsh);
    const float gh = 35.9f * eh / sqrtf(theta_half) + 3e-5f, gd = INV_PI_180 * ed + 3e-5f, gp = INV_PI_180 * ed / sd + 3e-5f;
    const float fh = ph - floorf(ph), fd = pd - floorf(pd), fp = pp - floorf(pp);
    if (!(fh > gh && fh < 1.f - gh && fd > gd && fd < 1.f - gd && fp > gp && fp < 1.f - gp)) return false;
    int ih = (int)ph, id = (int)pd, ip = (int)pp;
    if (ih >= 90) ih = 89;
    if (id >= 89) id = 89;
    if (ip >= 179) ip = 179;
    ind = ip + id * 180 + ih * 180 * 90;
    return true;
}
PTB_HD V3 merl_eval(const float* table, V3 wi, V3 wo, V3 N) {
    V3 t1 = get_tangent(N);
    V3 t2 = cross(t1, N);
    V3 wil = v3(dot(wi, t1), dot(wi, t2), dot(wi, N));
    V3 wol = v3(dot(wo, t1), dot(wo, t2), dot(wo, N));
    float thetai = acosf(wil.z);
    if ((double)thetai >= PTB_PI_D / 2) return v3(0, 0, 0);
    float thetao = acosf(wol.z);
    if ((double)thetao >= PTB_PI_D / 2) return v3(0, 0, 0);
    int ind;
    if (!merl_index_fast(wil, wol, ind)) {
        float phio = atan2f(wol.y, wol.x);
        if (phio < 0) phio = (float)((double)phio + 2 * PTB_PI_D);
        float phii = atan2f(wil.y, wil.x);
        if (phii < 0) phii = (float)((double)phii + 2 * PTB_PI_D);
        ind = merl_index((double)thetai, (double)phii, (double)thetao, (double)phio);
    }
    return v3(table[ind], table[ind + PTB_MERL_N], table[ind + 2 * PTB_MERL_N]);
}

// test hook (PTB_KAT_MERL_INDEX): both evaluations of the bin index for one pair of local directions
PTB_HD void merl_index_both(V3 wil, V3 wol, int& fast, int& exact) {
    fast = -1;
    int ind;
    if (merl_index_fast(wil, wol, ind)) fast = ind;
    float thetai = acosf(wil.z), thetao = acosf(wol.z);
    float phio = atan2f(wol.y, wol.x);
    if (phio < 0) phio = (float)((double)phio + 2 * PTB_PI_D);
    float phii = atan2f(wil.y, wil.x);
    if (phii < 0) phii = (float)((double)phii + 2 * PTB_PI_D);
    exact = merl_index((double)thetai, (double)phii, (double)thetao, (double)phio);
}

// ---- Texture lookups (BRDF.h:270-392): nearest texel, wrap -----------------------------------------
struct TexDev {
    float mult[3];
    int32_t W, H;        // W == 0: constant slot
    uint32_t offset;     // first float of the W*H*3 texels in the texel pool
};
PTB_HD float tex_wrap(float u) {
    u -= (float)(int)u;
    if (u < 0) u += 1;
    return u;
}
// non-finite uv never index a texture (SURVEY App. D#17: the reference reads out of bounds there)
PTB_HD int tex_index(const TexDev& t, float u, float v) {
    int x = (int)(u * (float)(t.W - 1));
    int y = (int)(v * (float)(t.H - 1));
    if (!(x >= 0)) x = 0;
    if (!(y >= 0)) y = 0;
    if (x > t.W - 1) x = t.W - 1;
    if (y > t.H - 1) y = t.H - 1;
    return (y * t.W + x) * 3;
}
PTB_HD V3 tex_vec(const TexDev& t, const float* pool, float u, float v) {
    if (t.W > 0) {
        const float* p = pool + t.offset + tex_index(t, u, v);
        return v3(p[0] * t.mult[0], p[1] * t.mult[1], p[2] * t.mult[2]);
    }
    return v3(t.mult[0], t.mult[1], t.mult[2]);
}
PTB_HD float tex_red(const TexDev& t, const float* pool, float u, float v) {
    if (t.W > 0) return pool[t.offset + tex_index(t, u, v)] * t.mult[0];
    return t.mult[0];
}
PTB_HD V3 tex_normal(const TexDev& t, const float* pool, float u, float v) {
    if (t.W > 0) {
        const float* p = pool + t.offset + tex_index(t, u, v);
        return v3(p[0], p[1], p[2]);
    }
    return v3(0.f, 0.f, 1.f);
}

// ---- Camera::generateDirection (Vector.h:792-825), non-lenticular, init_t = 0 ----------------------
struct CameraDev {
    V3 position, direction, up, right;  // right = cross(direction, up)
    float k;                            // W / (2 tan(fov/2))
    float focus_distance, aperture;
    int32_t W, H;
};
PTB_HD void camera_setup(CameraDev& c, const float* pos, const float* dir, const float* up, float fov, float focus,
                         float aperture, int W, int H) {
    c.position = v3(pos[0], pos[1], pos[2]);
    c.direction = v3(dir[0], dir[1], dir[2]);
    c.up = v3(up[0], up[1], up[2]);
    c.right = cross_rn(c.direction, c.up);
    c.k = (float)W / (2 * tanf(fov / 2));
    c.focus_distance = focus;
    c.aperture = aperture;
    c.W = W;
    c.H = H;
}
PTB_HD void camera_ray(const CameraDev& c, int i, int j, float dx, float dy, float ax, float ay, V3& o, V3& d) {
    // j - W/2 + 0.5 + dx : integer W/2, sum in double, narrowed to float by the Vector ctor
    // every operation rounded like the reference's (no FMA contraction): camera rays are BIT-IDENTICAL to generateDirection's, so a
    // primary ray that grazes an edge grazes it on the same side in both implementations
    V3 dv = v3((float)((double)(j - c.W / 2) + 0.5 + (double)dx), (float)((double)(i - c.H / 2) + 0.5 + (double)dy), c.k);
    dv = normalize_rn(dv);
    dv = add3_rn(add3_rn(scale_rn(dv.x, c.right), scale_rn(dv.y, c.up)), scale_rn(dv.z, c.direction));
    const V3 dest = add3_rn(c.position, scale_rn(div_rn(c.focus_distance, fabsf(dot_rn(dv, c.direction))), dv));
    o = add3_rn(add3_rn(c.position, scale_rn(ax, c.right)), scale_rn(ay, c.up));
    d = normalize_rn(sub3_rn(dest, o));
    // + init_t * d / dot(d, direction) with init_t == 0 (Scene::double_frustum_start_t)
    const float dd = dot_rn(d, c.direction);
    o = add3_rn(o, v3(div_rn(mul_rn(0.f, d.x), dd), div_rn(mul_rn(0.f, d.y), dd), div_rn(mul_rn(0.f, d.z), dd)));
}

// ---- pixel-filter tables (Raytracer.cpp:1354-1374) and the border ratio (1604-1609) -----------------
#define PTB_MAX_FILTER 4  /* filter_size = ceil(2 sigma) <= 4 */
struct FilterDev {
    int32_t size, width;                                   // filter_size, filter_total_width
    float integral[(2 * PTB_MAX_FILTER + 1) * (2 * PTB_MAX_FILTER + 1)];
    float sigma, denom2;                                   // denom2 = 1/(2 sigma^2)
};
inline void filter_setup(FilterDev& f, float sigma) {
    f.sigma = sigma;
    f.size = (int)ceilf(sigma * 2);
    f.width = 2 * f.size + 1;
    f.denom2 = 1.f / (2.f * sigma * sigma);
    for (int i = -f.size; i <= f.size; i++)
        for (int j = -f.size; j <= f.size; j++) {
            float integ = 0;
            for (int i2 = -f.size; i2 <= i; i2++)
                for (int j2 = -f.size; j2 <= j; j2++) {
                    float w = (float)(fast_exp(-(i2 * i2 + j2 * j2) / (2. * sigma * sigma)) / ((double)(sigma * sigma) * 2. * PTB_PI_D));
                    integ += w;
                }
            f.integral[(i + f.size) * f.width + (j + f.size)] = integ;
        }
}
PTB_HD float filter_sat(const float* sat, int w, int i0, int i1, int j0, int j1) {  // sum_area_table, Raytracer.cpp:1276-1291
    float t1 = 0, t2 = 0, t3 = 0;
    if (i0 > 0) t1 = sat[(i0 - 1) * w + j1];
    if (j0 > 0) t2 = sat[i1 * w + j0 - 1];
    if (i0 > 0 && j0 > 0) t3 = sat[(i0 - 1) * w + j0 - 1];
    return sat[i1 * w + j1] - t1 - t2 + t3;
}
PTB_HD float filter_ratio(const FilterDev& f, int i, int j, int W, int H, int& bmin_i, int& bmax_i, int& bmin_j, int& bmax_j) {
    bmin_i = i - f.size > 0 ? i - f.size : 0;
    bmax_i = i + f.size < H - 1 ? i + f.size : H - 1;
    bmin_j = j - f.size > 0 ? j - f.size : 0;
    bmax_j = j + f.size < W - 1 ? j + f.size : W - 1;
    return div_rn(1.f, filter_sat(f.integral, f.width, bmin_i - i + f.size, bmax_i - i + f.size, bmin_j - j + f.size, bmax_j - j + f.size));   // bit-exact block: IEEE division whatever -prec-div says
}
// splat weight of sample (i,j,dx,dy) into pixel (i2,j2), Raytracer.cpp:1652
PTB_HD float filter_weight(const FilterDev& f, float denom1, int i2, int j2, int i, int j, float dx, float dy) {
    float a = (float)(i2 - i) - dy, b = (float)(j2 - j) - dx;
    float e = -(a * a + b * b) * f.denom2;
    return (float)(fast_exp((double)e) * (double)denom1);
}

}  // namespace ptb
