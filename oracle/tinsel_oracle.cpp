// oracle/tinsel_oracle.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// CPU restatement ("port") of tinsel's one data-parallel hot path, in plain scalar C++ over the
// C-ABI scene description (include/tinsel_b200.h): per-sample camera ray, two-level BVH closest
// hit with sphere / plane / two-sided triangle tests, Disney BSDF eval / pdf / sample, MIS
// next-event estimation against the HDR probe and area lights, Beer-Lambert media, sky, and the
// Gaussian / box filtered accumulation.  Every function cites the reference file:line it
// follows (paths under /root/reference/src).  It walks the reference's ORIGINAL data layout
// (32-byte BVHNode arrays, index + vertex arrays) -- unlike the CUDA path, which re-packs both --
// so agreement between the two also checks the re-layout.
//
// Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / reference arms may load this
// library.  Parity pin: tests/test_oracle.py checks it bit-for-bit, per sample, against
// oracle/_ref/libtinsel_ref_detmath.so (the reference's own src/render.cpp compiled with the
// same deterministic libm, include/tb200_detmath.h) and against tests/golden/*.npz produced by
// that library (tools/make_golden.py).
//
// Arithmetic rules: fp32 evaluated left to right exactly as the cited expression; the reference's
// implicit double promotions are kept where they change the result (material constants) and are
// written as fp32 where double rounding is provably innocuous (a single /, +, sqrt of floats).
// Build: -O2 -ffp-contract=off, no -ffast-math (oracle/Makefile).
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <thread>
#include <vector>
#include <algorithm>

#include "tb200_detmath.h"
#include "tinsel_b200.h"

// -DTB_ORACLE_LIBM (libtinsel_oracle_libm.so): the transcendentals come from the system libm, as in the
// reference as shipped (the "literal" flavour of oracle/_ref); the default build uses the deterministic
// ones the kernels use, so only this flavour may differ from the CUDA path, in the last bits.
#ifdef TB_ORACLE_LIBM
#define tbm_sinf sinf
#define tbm_cosf cosf
#define tbm_expf expf
#define tbm_powf powf
#define tbm_acosf acosf
#define tbm_atan2f atan2f
#endif

// Optional work counters (-DTB_ORACLE_COUNT, built as libtinsel_oracle_count.so): the inputs of the
// ALGORITHMIC-bytes formula of SURVEY.md 8(d), counted on the reference traversal order.
enum { C_VINT, C_TTRI, C_TPRIM, C_HMESH, C_HIT, C_NEE_BYTES, C_PROBE_BYTES, C_MISS_BYTES, C_FB_PIXELS, C_RAYS, C_SAMPLES, C_NUM };
#ifdef TB_ORACLE_COUNT
#include <atomic>
static std::atomic<unsigned long long> g_counters[C_NUM];
#define COUNT(which, n) g_counters[which].fetch_add((unsigned long long)(n), std::memory_order_relaxed)
#else
#define COUNT(which, n) ((void)0)
#endif

namespace {

struct vec3 {
    float x, y, z;
};

inline vec3 mk(float x, float y, float z) { return vec3{x, y, z}; }
inline vec3 splat(float s) { return vec3{s, s, s}; }
inline vec3 from(const float* f) { return vec3{f[0], f[1], f[2]}; }
inline vec3 add(vec3 a, vec3 b) { return mk(a.x + b.x, a.y + b.y, a.z + b.z); }
inline vec3 sub(vec3 a, vec3 b) { return mk(a.x - b.x, a.y - b.y, a.z - b.z); }
inline vec3 scale(vec3 a, float s) { return mk(a.x * s, a.y * s, a.z * s); }
inline vec3 mul(vec3 a, vec3 b) { return mk(a.x * b.x, a.y * b.y, a.z * b.z); }
inline vec3 neg(vec3 a) { return mk(-a.x, -a.y, -a.z); }
// Vec3 / Real is a*(1.0/s) (maths.h:242); one double division rounds to float like 1.0f/s
inline vec3 divs(vec3 a, float s) { return scale(a, 1.0f / s); }
inline float dot3(vec3 a, vec3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }                           // maths.h:257
inline vec3 cross3(vec3 a, vec3 b) { return mk(a.y * b.z - b.y * a.z, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }  // maths.h:256
inline float len3(vec3 a) { return sqrtf(dot3(a, a)); }
inline vec3 unit(vec3 a) { return divs(a, len3(a)); }                                                       // maths.h:260
inline vec3 safe_unit(vec3 a, vec3 fallback)                                                               // maths.h:261-273
{
    float m = dot3(a, a);
    return m > 0.0f ? scale(a, 1.0f / sqrtf(m)) : fallback;
}
inline float fmin2(float a, float b) { return a < b ? a : b; }        // Min, maths.h:56
inline float fmax2(float a, float b) { return a < b ? b : a; }        // Max, maths.h:59
inline int imin2(int a, int b) { return a < b ? a : b; }
inline int imax2(int a, int b) { return a < b ? b : a; }
inline float clampf(float x, float lo, float hi) { return fmin2(fmax2(x, lo), hi); }   // maths.h:62-66
inline int clampi(int x, int lo, int hi) { return imin2(imax2(x, lo), hi); }
inline float absf(float x) { return x < 0.0f ? -x : x; }              // Abs, maths.h:68-75
inline float mixf(float a, float b, float t) { return a + (b - a) * t; }   // Lerp, maths.h:79-83
inline vec3 mix3(vec3 a, vec3 b, float t) { return add(a, scale(sub(b, a), t)); }
inline vec3 face_fwd(vec3 n, vec3 v) { return dot3(v, n) < 0.0f ? neg(n) : n; }   // maths.h:1591-1598

const float PI = 3.141592653589793f;        // kPi, maths.h:32
const float TWO_PI = 3.141592653589793f * 2.0f;
const float INV_PI = 1.0f / PI;
const float INV_2PI = 1.0f / TWO_PI;
const float RAY_EPS = 0.0001f;              // kRayEpsilon, render.cpp:11

struct quat {
    float x, y, z, w;
};
inline quat qmul(quat a, quat b)   // maths.h:531-537
{
    return quat{a.w * b.x + b.w * a.x + a.y * b.z - b.y * a.z, a.w * b.y + b.w * a.y + a.z * b.x - b.z * a.x,
                a.w * b.z + b.w * a.z + a.x * b.y - b.x * a.y, a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z};
}
inline quat qconj(quat q) { return quat{-q.x, -q.y, -q.z, q.w}; }
inline vec3 qrot(quat q, vec3 v)   // Rotate, maths.h:558-563
{
    quat t = qmul(qmul(q, quat{v.x, v.y, v.z, 0.0f}), qconj(q));
    return mk(t.x, t.y, t.z);
}

struct xform {
    vec3 p;
    quat r;
    float s;
};
inline xform xf_from(const tb200_transform& t) { return xform{from(t.p), quat{t.r[0], t.r[1], t.r[2], t.r[3]}, t.s}; }
// InterpolateTransform, maths.h:1566-1569 (Quat Lerp + Normalize(Quat) maths.h:547-553)
inline xform xf_lerp(const xform& a, const xform& b, float t)
{
    xform r;
    r.p = add(a.p, scale(sub(b.p, a.p), t));
    quat q{a.r.x + (b.r.x - a.r.x) * t, a.r.y + (b.r.y - a.r.y) * t, a.r.z + (b.r.z - a.r.z) * t, a.r.w + (b.r.w - a.r.w) * t};
    float len = sqrtf(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w);
    float rcp = 1.0f / len;
    r.r = quat{q.x * rcp, q.y * rcp, q.z * rcp, q.w * rcp};
    r.s = a.s + (b.s - a.s) * t;
    return r;
}
inline vec3 xf_vector(const xform& t, vec3 v) { return qrot(t.r, scale(v, t.s)); }                    // maths.h:601
inline vec3 xf_point(const xform& t, vec3 v) { return add(t.p, qrot(t.r, scale(v, t.s))); }           // maths.h:606
inline vec3 xf_inv_vector(const xform& t, vec3 v) { return scale(qrot(qconj(t.r), v), 1.0f / t.s); }  // maths.h:611
inline vec3 xf_inv_point(const xform& t, vec3 v) { return scale(qrot(qconj(t.r), sub(v, t.p)), 1.0f / t.s); }  // maths.h:616

// ---- Random, maths.h:1036-1091 ---------------------------------------------------------------
struct rng_t {
    uint32_t a, b;
};
inline rng_t rng_make(uint32_t seed)
{
    rng_t r;
    r.a = 315645664u + seed;
    r.b = r.a ^ 0x13ab45feu;
    return r;
}
inline uint32_t rng_u32(rng_t& r)
{
    uint32_t a = r.a, b = r.b;
    r.a = (b ^ ((a << 5) | (a >> 27))) ^ (a * b);
    r.b = r.a ^ ((b << 12) | (b >> 20));
    return r.a;
}
inline float rng_f(rng_t& r) { return (float)rng_u32(r) * (1.0f / (float)0xffffffffu); }

// ---- scene access --------------------------------------------------------------------------------
struct Oracle {
    const tb200_scene* scene;
};

inline bool node_is_leaf(const tb200_bvh_node& n) { return (n.right_leaf >> 31) != 0; }
inline uint32_t node_right(const tb200_bvh_node& n) { return n.right_leaf & 0x7fffffffu; }

// IntersectRayAABBFast, intersection.h:373-397
inline bool slab(vec3 pos, vec3 rcp, const float* lo, const float* hi, float& t)
{
    float l1 = (lo[0] - pos.x) * rcp.x, l2 = (hi[0] - pos.x) * rcp.x;
    float lmin = l1 < l2 ? l1 : l2, lmax = l1 > l2 ? l1 : l2;
    l1 = (lo[1] - pos.y) * rcp.y;
    l2 = (hi[1] - pos.y) * rcp.y;
    float mn = l1 < l2 ? l1 : l2, mx = l1 > l2 ? l1 : l2;
    lmin = mn > lmin ? mn : lmin;
    lmax = mx < lmax ? mx : lmax;
    l1 = (lo[2] - pos.z) * rcp.z;
    l2 = (hi[2] - pos.z) * rcp.z;
    mn = l1 < l2 ? l1 : l2;
    mx = l1 > l2 ? l1 : l2;
    lmin = mn > lmin ? mn : lmin;
    lmax = mx < lmax ? mx : lmax;
    bool hit = (lmax >= 0.f) & (lmax >= lmin);
    if (hit) t = lmin;
    return hit;
}

// IntersectRayTriTwoSided, intersection.h:117-145
inline bool tri_two_sided(vec3 p, vec3 dir, vec3 a, vec3 b, vec3 c, float& t, float& u, float& v, float& w, float& sign, vec3& n)
{
    vec3 ab = sub(b, a), ac = sub(c, a);
    vec3 nn = cross3(ab, ac);
    float d = dot3(neg(dir), nn);
    float ood = 1.0f / d;
    vec3 ap = sub(p, a);
    t = dot3(ap, nn) * ood;
    if (t < 0.0f) return false;
    vec3 e = cross3(neg(dir), ap);
    v = dot3(ac, e) * ood;
    if (v < 0.0f || v > 1.0f) return false;
    w = -dot3(ab, e) * ood;
    if (w < 0.0f || v + w > 1.0f) return false;
    u = 1.0f - v - w;
    n = nn;
    sign = d;
    return true;
}

struct mesh_hit {
    float t, u, v, w;
    int tri;
    vec3 n;
};

// IntersectRayMesh + MeshQuery, intersection.h:629-749
bool mesh_closest(const tb200_mesh& m, vec3 o, vec3 d, mesh_hit& out)
{
    vec3 rcp = mk(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
    int stack[32];
    stack[0] = 0;
    int count = 1;
    float closest = FLT_MAX, tmax = FLT_MAX;
    while (count) {
        const tb200_bvh_node& node = m.nodes[stack[--count]];
        if (node_is_leaf(node)) {
            COUNT(C_TTRI, 1);
            int i = (int)node.left;
            int i0 = m.indices[i * 3 + 0], i1 = m.indices[i * 3 + 1], i2 = m.indices[i * 3 + 2];
            float t, u, v, w, sign;
            vec3 n;
            if (tri_two_sided(o, d, from(m.positions + 3 * i0), from(m.positions + 3 * i1), from(m.positions + 3 * i2), t, u, v, w, sign, n)) {
                if (t > 0.0f && t < closest) {
                    closest = t;
                    out.u = u;
                    out.v = v;
                    out.w = w;
                    out.tri = i;
                    out.n = scale(n, sign);
                }
            }
            tmax = closest;
        } else {
            COUNT(C_VINT, 1);
            uint32_t li = node.left, ri = node_right(node);
            const tb200_bvh_node& L = m.nodes[li];
            const tb200_bvh_node& R = m.nodes[ri];
            float tl, tr;
            bool hl = slab(o, rcp, L.lower, L.upper, tl) && tl < tmax;
            bool hr = slab(o, rcp, R.lower, R.upper, tr) && tr < tmax;
            if (hl && hr && tl < tr) {
                uint32_t tmp = li;
                li = ri;
                ri = tmp;
            }
            if (hl) stack[count++] = (int)li;
            if (hr) stack[count++] = (int)ri;
        }
    }
    if (closest < FLT_MAX) {
        out.t = closest;
        return true;
    }
    return false;
}

// IntersectRaySphere + SolveQuadratic, intersection.h:30-83
bool sphere_hit(vec3 center, float radius, vec3 o, vec3 d, float& tOut, vec3& nOut)
{
    vec3 q = sub(o, center);
    float a = 1.0f;
    float b = 2.0f * dot3(q, d);
    float c = dot3(q, q) - (radius * radius);
    float disc = b * b - 4.0f * a * c;
    if (disc < 0.0f) return false;
    float t = -0.5f * (b + (b < 0.0f ? -1.0f : 1.0f) * sqrtf(disc));
    float mn = t / a, mx = c / t;
    if (mx < mn) {
        float s = mn;
        mn = mx;
        mx = s;
    }
    if (mn < 0.0f && mx < 0.0f) return false;
    if (mn < 0.0f && mx > 0.0f) mn = mx;
    nOut = unit(sub(add(o, scale(d, mn)), center));
    tOut = mn;
    return true;
}

// PrimitiveIntersect, intersection.h:951-1020
bool prim_hit(const tb200_scene& sc, const tb200_primitive& p, vec3 o, vec3 d, float time, float& tOut, vec3& nOut)
{
    xform xf = xf_lerp(xf_from(p.start), xf_from(p.end), time);
    if (p.type == TB200_SPHERE) return sphere_hit(xf.p, p.radius * xf.s, o, d, tOut, nOut);
    if (p.type == TB200_PLANE) {
        // IntersectRayPlane, intersection.h:85-99
        float dd = p.plane[0] * d.x + p.plane[1] * d.y + p.plane[2] * d.z + p.plane[3] * 0.0f;
        if (dd == 0.0f) return false;
        float t = -(p.plane[0] * o.x + p.plane[1] * o.y + p.plane[2] * o.z + p.plane[3] * 1.0f) / dd;
        tOut = t;
        nOut = mk(p.plane[0], p.plane[1], p.plane[2]);
        return t > 0.0f;
    }
    const tb200_mesh& m = sc.meshes[p.mesh];
    vec3 lo = xf_inv_point(xf, o), ld = xf_inv_vector(xf, d);
    mesh_hit mh;
    if (!mesh_closest(m, lo, ld, mh)) return false;
    COUNT(C_HMESH, 1);
    int i0 = m.indices[mh.tri * 3 + 0], i1 = m.indices[mh.tri * 3 + 1], i2 = m.indices[mh.tri * 3 + 2];
    vec3 n1 = from(m.normals + 3 * i0), n2 = from(m.normals + 3 * i1), n3 = from(m.normals + 3 * i2);
    vec3 smooth = add(add(scale(n1, mh.u), scale(n2, mh.v)), scale(n3, mh.w));
    if (dot3(smooth, mh.n) < 0.0f) smooth = scale(smooth, -1.0f);
    tOut = mh.t;
    nOut = safe_unit(xf_vector(xf, smooth), mh.n);
    return true;
}

struct hit_t {
    float t;
    vec3 n;
    int prim;
};

// Trace + QueryBVH, render.cpp:17-62, intersection.h:751-799
hit_t closest_hit(const tb200_scene& sc, vec3 o, vec3 d, float time)
{
    COUNT(C_RAYS, 1);
    vec3 rcp = mk(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
    int stack[32];
    stack[0] = 0;
    int count = 1;
    float minT = FLT_MAX;
    int best = -1;
    vec3 bestN = splat(0.0f);
    while (count) {
        const tb200_bvh_node& node = sc.bvhNodes[stack[--count]];
        if (node_is_leaf(node)) {
            COUNT(C_TPRIM, 1);
            float t;
            vec3 n = splat(0.0f);
            if (prim_hit(sc, sc.primitives[node.left], o, d, time, t, n)) {
                if (t < minT && t > 0.0f) {
                    minT = t;
                    best = (int)node.left;
                    bestN = n;
                }
            }
        } else {
            COUNT(C_VINT, 1);
            uint32_t li = node.left, ri = node_right(node);
            const tb200_bvh_node& L = sc.bvhNodes[li];
            const tb200_bvh_node& R = sc.bvhNodes[ri];
            float tl, tr;
            bool hl = slab(o, rcp, L.lower, L.upper, tl);
            bool hr = slab(o, rcp, R.lower, R.upper, tr);
            if (hl && hr && tl < tr) {
                uint32_t tmp = li;
                li = ri;
                ri = tmp;
            }
            if (hl) stack[count++] = (int)li;
            if (hr) stack[count++] = (int)ri;
        }
    }
    hit_t h;
    h.t = minT;
    h.prim = best;
    h.n = face_fwd(bestN, neg(d));
    return h;
}

// ---- Disney BSDF, disney.h -------------------------------------------------------------------------

inline float mat_ior(const tb200_material& m)   // Material::GetIndexOfRefraction, scene.h:72-78
{
    if (m.eta == 0.0f) return 2.0f / (1.0f - sqrtf((float)(0.08 * (double)m.specular))) - 1.0f;
    return m.eta;
}
inline float schlick(float u)   // disney.h:49-54
{
    float m = clampf(1 - u, 0.0f, 1.0f);
    float m2 = m * m;
    return m2 * m2 * m;
}
inline float gtr1(float NDotH, float a)   // disney.h:56-62
{
    if (a >= 1) return INV_PI;
    float a2 = a * a;
    float t = 1 + (a2 - 1) * NDotH * NDotH;
    return (a2 - 1) / (PI * logf(a2) * t);
}
inline float gtr2(float NDotH, float a)   // disney.h:64-69
{
    float a2 = a * a;
    float t = 1.0f + (a2 - 1.0f) * NDotH * NDotH;
    return a2 / (PI * t * t);
}
inline float smith(float NDotv, float alphaG)   // disney.h:71-76
{
    float a = alphaG * alphaG;
    float b = NDotv * NDotv;
    return 1 / (NDotv + sqrtf(a + b - a * b));
}
inline float fresnel(float VDotN, float etaI, float etaT)   // Fr, disney.h:79-96
{
    float q = etaI / etaT;
    float s2 = (q * q) * (1.0f - VDotN * VDotN);
    if (s2 > 1.0f) return 1.0f;
    float LDotN = sqrtf(1.0f - s2);
    float eta = etaT / etaI;
    float r1 = (VDotN - eta * LDotN) / (VDotN + eta * LDotN);
    float r2 = (LDotN - eta * VDotN) / (LDotN + eta * VDotN);
    return 0.5f * (r1 * r1 + r2 * r2);
}

// BSDFPdf, disney.h:125-166
float bsdf_pdf(const tb200_material& mat, float etaI, float etaO, vec3 n, vec3 V, vec3 L)
{
    if (dot3(L, n) <= 0.0f) {
        float bsdfPdf = 0.0f;
        float brdfPdf = INV_2PI * mat.subsurface * 0.5f;
        return mixf(brdfPdf, bsdfPdf, mat.transmission);
    }
    float F = fresnel(dot3(n, V), etaI, etaO);
    float a = fmax2(0.001f, mat.roughness);
    vec3 half = safe_unit(add(L, V), splat(0.0f));
    float cosThetaHalf = absf(dot3(half, n));
    float pdfHalf = gtr2(cosThetaHalf, a) * cosThetaHalf;
    float pdfSpec = 0.25f * pdfHalf / fmax2(1.e-6f, dot3(L, half));
    float pdfDiff = absf(dot3(L, n)) * INV_PI * (1.0f - mat.subsurface);
    float bsdfPdf = pdfSpec * F;
    float brdfPdf = mixf(pdfDiff, pdfSpec, 0.5f);
    return mixf(brdfPdf, bsdfPdf, mat.transmission);
}

// BSDFEval, disney.h:296-405 (double intermediates kept where the reference has them)
vec3 bsdf_eval(const tb200_material& mat, float etaI, float etaO, vec3 N, vec3 V, vec3 L)
{
    float NDotL = dot3(N, L), NDotV = dot3(N, V);
    vec3 H = unit(add(L, V));
    float NDotH = dot3(N, H), LDotH = dot3(L, H);

    vec3 Cdlin = from(mat.color);
    float Cdlum = (float)(.3 * (double)Cdlin.x + .6 * (double)Cdlin.y + .1 * (double)Cdlin.z);
    vec3 Ctint = Cdlum > 0.0f ? divs(Cdlin, Cdlum) : splat(1.0f);
    float spec08 = (float)((double)mat.specular * .08);
    vec3 Cspec0 = mix3(scale(mix3(splat(1.0f), Ctint, mat.specularTint), spec08), Cdlin, mat.metallic);

    vec3 bsdf = splat(0.0f), brdf = splat(0.0f);
    if (mat.transmission > 0.0f) {
        if (NDotL <= 0) {
            float F = fresnel(NDotV, etaI, etaO);
            bsdf = splat(mat.transmission * (1.0f - F) / absf(NDotL) * (1.0f - mat.metallic));
        } else {
            float a = fmax2(0.001f, mat.roughness);
            float Ds = gtr2(NDotH, a);
            float FH = fresnel(LDotH, etaI, etaO);
            vec3 Fs = mix3(Cspec0, splat(1.0f), FH);
            float Gs = smith(NDotV, a) * smith(NDotL, a);
            bsdf = scale(scale(Fs, Gs), Ds);
        }
    }
    if (mat.transmission < 1.0f) {
        if (NDotL <= 0) {
            if (mat.subsurface > 0.0f) {
                vec3 s = mk(sqrtf(mat.color[0]), sqrtf(mat.color[1]), sqrtf(mat.color[2]));
                float FL = schlick(absf(NDotL)), FV = schlick(NDotV);
                float Fd = (1.0f - 0.5f * FL) * (1.0f - 0.5f * FV);
                brdf = scale(scale(scale(scale(s, INV_PI), mat.subsurface), Fd), 1.0f - mat.metallic);
            }
        } else {
            float a = fmax2(0.001f, mat.roughness);
            float Ds = gtr2(NDotH, a);
            float FH = schlick(LDotH);
            vec3 Fs = mix3(Cspec0, splat(1.0f), FH);
            float Gs = smith(NDotV, a) * smith(NDotL, a);
            float FL = schlick(NDotL), FV = schlick(NDotV);
            float Fd90 = (float)(0.5 + (double)(2.0f * LDotH * LDotH * mat.roughness));
            float Fd = mixf(1.0f, Fd90, FL) * mixf(1.0f, Fd90, FV);
            float Dr = gtr1(NDotH, (float)(.1 + (.001 - .1) * (double)mat.clearcoatGloss));
            float Fc = mixf(.04f, 1.0f, FH);
            float Gr = smith(NDotL, .25f) * smith(NDotV, .25f);
            vec3 diffuse = scale(scale(scale(Cdlin, INV_PI * Fd), 1.0f - mat.metallic), 1.0f - mat.subsurface);
            vec3 spec = scale(scale(Fs, Gs), Ds);
            brdf = add(add(diffuse, spec), splat(mat.clearcoat * Gr * Fc * Dr));
        }
    }
    return mix3(brdf, bsdf, mat.transmission);
}

// BasisFromVector, maths.h:1261-1275
void basis(vec3 w, vec3& u, vec3& v)
{
    if (fabsf(w.x) > fabsf(w.y)) {
        float inv = 1.0f / sqrtf(w.x * w.x + w.z * w.z);
        u = mk(-w.z * inv, 0.0f, w.x * inv);
    } else {
        float inv = 1.0f / sqrtf(w.y * w.y + w.z * w.z);
        u = mk(0.0f, w.z * inv, -w.y * inv);
    }
    v = cross3(w, u);
}

vec3 ggx_reflect(const tb200_material& mat, float r1, float r2, vec3 U, vec3 Vt, vec3 N, vec3 view)   // disney.h:183-205
{
    float a = fmax2(0.001f, mat.roughness);
    float phi = r1 * TWO_PI;
    float ct = sqrtf((1.0f - r2) / (1.0f + (a * a - 1.0f) * r2));
    float st = sqrtf(fmax2(0.0f, 1.0f - ct * ct));
    float sp = tbm_sinf(phi), cp = tbm_cosf(phi);
    vec3 half = add(add(scale(U, st * cp), scale(Vt, st * sp)), scale(N, ct));
    if (dot3(half, view) <= 0.0f) half = scale(half, -1.0f);
    return sub(scale(half, 2.0f * dot3(view, half)), view);
}

enum { REFLECTED = 0, TRANSMITTED = 1, SPECULAR = 2 };

// BSDFSample, disney.h:170-293
void bsdf_sample(const tb200_material& mat, float etaI, float etaO, vec3 U, vec3 Vt, vec3 N, vec3 view, vec3& light, float& pdf,
                 int& type, rng_t& rng)
{
    if (rng_f(rng) < mat.transmission) {
        float F = fresnel(dot3(N, view), etaI, etaO);
        if (rng_f(rng) < F) {
            float r1 = rng_f(rng), r2 = rng_f(rng);
            type = REFLECTED;
            light = ggx_reflect(mat, r1, r2, U, Vt, N, view);
        } else {
            // Refract, disney.h:34-47
            float eta = etaI / etaO;
            float ci = dot3(N, view);
            float s2i = fmax2(0.0f, 1.0f - ci * ci);
            float s2t = eta * eta * s2i;
            if (s2t >= 1) {
                pdf = 0.0f;
                return;
            }
            float ctt = sqrtf(1.0f - s2t);
            light = add(scale(neg(view), eta), scale(N, eta * ci - ctt));
            type = SPECULAR;
            pdf = (1.0f - F) * mat.transmission;
            return;
        }
    } else {
        float r1 = rng_f(rng), r2 = rng_f(rng);
        if (rng_f(rng) < 0.5f) {
            if (rng_f(rng) < mat.subsurface) {
                // UniformSampleHemisphere, maths.h:1291-1302
                float z = rng_f(rng);
                float w = sqrtf(1.0f - z * z);
                float phi = TWO_PI * rng_f(rng);
                float x = tbm_cosf(phi) * w, y = tbm_sinf(phi) * w;
                light = sub(add(scale(U, x), scale(Vt, y)), scale(N, z));
                type = TRANSMITTED;
            } else {
                // CosineSampleHemisphere via UniformSampleDisc, maths.h:1304-1325
                float r = sqrtf(r1);
                float th = TWO_PI * r2;
                float sx = r * tbm_cosf(th), sy = r * tbm_sinf(th);
                float z = sqrtf(fmax2(0.0f, 1.0f - sx * sx - sy * sy));
                light = add(add(scale(U, sx), scale(Vt, sy)), scale(N, z));
                type = REFLECTED;
            }
        } else {
            light = ggx_reflect(mat, r1, r2, U, Vt, N, view);
            type = REFLECTED;
        }
    }
    pdf = bsdf_pdf(mat, etaI, etaO, N, view, light);
}

// ---- probe / sky, probe.h + scene.h:161-181 --------------------------------------------------------

void dir_to_uv(vec3 d, float& u, float& v)   // probe.h:105-113
{
    float theta = tbm_acosf(clampf(d.y, -1.0f, 1.0f));
    float phi = (d.x == 0.0f && d.z == 0.0f) ? 0.0f : tbm_atan2f(d.z, d.x);
    u = (PI + phi) * INV_PI * 0.5f;
    v = theta * INV_PI;
}

float probe_pdf(const tb200_sky& s, vec3 d)   // probe.h:136-160
{
    float u, v;
    dir_to_uv(d, u, v);
    int col = clampi(int(u * s.probeWidth), 0, s.probeWidth - 1);
    int row = clampi(int(v * s.probeHeight), 0, s.probeHeight - 1);
    float pdf = s.pdfValuesX[row * s.probeWidth + col] * s.pdfValuesY[row];
    float sinTheta = tbm_sinf(v * PI);
    if (fabsf(sinTheta) < 0.0001f)
        pdf = 0.0f;
    else
        pdf *= float(s.probeWidth) * float(s.probeHeight) / (2.0f * PI * PI * sinTheta);
    return pdf;
}

int lower_bound(const float* a, int lo, int hi, float value)   // probe.h:186-203
{
    while (lo < hi) {
        int mid = lo + (hi - lo) / 2;
        if (a[mid] < value)
            lo = mid + 1;
        else
            hi = mid;
    }
    return lo;
}

void probe_sample(const tb200_sky& s, vec3& dir, vec3& color, float& pdf, rng_t& rng)   // probe.h:205-236
{
    float r1 = rng_f(rng), r2 = rng_f(rng);
    int W = s.probeWidth, H = s.probeHeight;
    {
        int lw = 0, lh = 0;
        while ((1 << lw) < W) ++lw;
        while ((1 << lh) < H) ++lh;
        COUNT(C_PROBE_BYTES, 4 * (lw + lh) + 24);
    }
    int row = lower_bound(s.cdfValuesY, 0, H, r1);
    int col = lower_bound(s.cdfValuesX, row * W, (row + 1) * W, r2) - row * W;
    color = from(s.probeData + 4 * (size_t)(row * W + col));
    pdf = s.pdfValuesX[row * W + col] * s.pdfValuesY[row];
    float u = col / float(W), v = row / float(H);
    float sinTheta = tbm_sinf(v * PI);
    if (sinTheta == 0.0f)
        pdf = 0.0f;
    else
        pdf *= (W * H) / (2.0f * PI * PI * sinTheta);
    float theta = v * PI, phi = u * 2.0f * PI;   // ProbeUVToDir, probe.h:115-125
    dir = mk(-tbm_sinf(theta) * tbm_cosf(phi), tbm_cosf(theta), -tbm_sinf(theta) * tbm_sinf(phi));
}

vec3 sky_eval(const tb200_sky& s, vec3 d)   // Sky::Eval scene.h:168-178, ProbeEval probe.h:128-134
{
    if (s.probeValid) {
        float u, v;
        dir_to_uv(d, u, v);
        int px = clampi(int(u * s.probeWidth), 0, s.probeWidth - 1);
        int py = clampi(int(v * s.probeHeight), 0, s.probeHeight - 1);
        return from(s.probeData + 4 * (size_t)(py * s.probeWidth + px));
    }
    return mix3(from(s.horizon), from(s.zenith), sqrtf(absf(d.y)));
}

// ---- lights, intersection.h:833-904 ----------------------------------------------------------------

float prim_area(const tb200_scene& sc, const tb200_primitive& p)   // PrimitiveArea
{
    if (p.type == TB200_SPHERE) return 4.0f * PI * p.radius * p.radius;
    if (p.type == TB200_MESH) return sc.meshes[p.mesh].area * p.end.s;
    return 0.0f;
}

void prim_sample(const tb200_scene& sc, const tb200_primitive& p, float time, vec3& pos, vec3& normal, rng_t& rng)   // PrimitiveSample
{
    xform xf = xf_lerp(xf_from(p.start), xf_from(p.end), time);
    if (p.type == TB200_SPHERE) {
        float u1 = rng_f(rng), u2 = rng_f(rng);
        // UniformSampleSphere, maths.h:1278-1287
        float z = 1.f - 2.f * u1;
        float r = sqrtf(fmax2(0.f, 1.f - z * z));
        float phi = 2.f * PI * u2;
        vec3 s = mk(r * tbm_cosf(phi), r * tbm_sinf(phi), z);
        pos = xf_point(xf, scale(s, p.radius));
        normal = unit(sub(pos, xf.p));
        return;
    }
    if (p.type == TB200_MESH) {
        const tb200_mesh& m = sc.meshes[p.mesh];
        int ntri = m.numIndices / 3;
        float r = rng_f(rng);
        int tri = imin2(lower_bound(m.cdf, 0, ntri, r), ntri - 1);
        float sr = sqrtf(rng_f(rng));   // UniformSampleTriangle, maths.h:1312-1317
        float u = 1.0f - sr;
        float v = rng_f(rng) * sr;
        int i0 = m.indices[tri * 3 + 0], i1 = m.indices[tri * 3 + 1], i2 = m.indices[tri * 3 + 2];
        vec3 a = from(m.positions + 3 * i0), b = from(m.positions + 3 * i1), c = from(m.positions + 3 * i2);
        vec3 n1 = from(m.normals + 3 * i0), n2 = from(m.normals + 3 * i1), n3 = from(m.normals + 3 * i2);
        float w = 1.0f - u - v;
        pos = xf_point(xf, add(add(scale(a, u), scale(b, v)), scale(c, w)));
        normal = safe_unit(xf_vector(xf, add(add(scale(n1, u), scale(n2, v)), scale(n3, w))), splat(0.0f));
        return;
    }
    pos = normal = splat(0.0f);
}

// SampleLights, render.cpp:103-227
vec3 sample_lights(const tb200_scene& sc, const tb200_primitive& surf, float etaI, float etaO, vec3 p, vec3 n, vec3 wo, float time,
                   rng_t& rng)
{
    vec3 sum = splat(0.0f);
    if (sc.sky.probeValid) {
        vec3 wi, skyColor;
        float skyPdf;
        probe_sample(sc.sky, wi, skyColor, skyPdf, rng);
        hit_t sh = closest_hit(sc, add(p, scale(face_fwd(n, wi), RAY_EPS)), wi, time);
        if (sh.prim < 0) {
            float bp = bsdf_pdf(surf.material, etaI, etaO, n, wo, wi);
            vec3 f = bsdf_eval(surf.material, etaI, etaO, n, wo, wi);
            if (bp > 0.0f) {
                float cbsdf = 1.0f / 2, csky = 1.0f / 2;
                float weight = csky * skyPdf / (cbsdf * bp + csky * skyPdf);
                if (weight > 0.0f) sum = add(sum, divs(scale(mul(scale(skyColor, weight), f), absf(dot3(wi, n))), skyPdf));
            }
        }
        sum = scale(sum, 1.0f);   // sum /= float(kProbeSamples)
    }
    for (int i = 0; i < sc.numPrimitives; ++i) {
        const tb200_primitive& light = sc.primitives[i];
        int numSamples = light.lightSamples;
        if (numSamples == 0) continue;
        vec3 L = splat(0.0f);
        for (int s = 0; s < numSamples; ++s) {
            vec3 lightPos, lightNormal;
            prim_sample(sc, light, time, lightPos, lightNormal, rng);
            {
                int extra = 0;
                if (light.type == TB200_MESH) {
                    int ntri = sc.meshes[light.mesh].numIndices / 3, l2 = 0;
                    while ((1 << l2) < ntri) ++l2;
                    extra = 4 * l2 + 84;
                }
                COUNT(C_NEE_BYTES, 136 + extra);
            }
            vec3 wi = sub(lightPos, p);
            float dSq = dot3(wi, wi);
            wi = divs(wi, sqrtf(dSq));
            hit_t sh = closest_hit(sc, add(p, scale(face_fwd(n, wi), RAY_EPS)), wi, time);
            if (sh.prim < 0) continue;
            float t = sh.t, tSq = t * t;
            if (!(fabsf(t - sqrtf(dSq)) <= 1.e-2f)) continue;
            float nl = absf(dot3(lightNormal, wi));
            if (absf(nl) < 1.e-6f) continue;
            float lightPdf = ((1.0f / prim_area(sc, light)) * tSq) / nl;
            float bp = bsdf_pdf(surf.material, etaI, etaO, n, wo, wi);
            vec3 f = bsdf_eval(surf.material, etaI, etaO, n, wo, wi);
            if (bp > 0.0f) {
                int N = int(light.lightSamples + 1.0f);
                float cbsdf = 1.0f / N, clight = float(light.lightSamples) / N;
                float weight = clight * lightPdf / (cbsdf * bp + clight * lightPdf);
                vec3 e = from(sc.primitives[sh.prim].material.emission);
                L = add(L, scale(mul(scale(f, weight), e), absf(dot3(wi, n)) / fmax2(1.e-3f, lightPdf)));
            }
        }
        sum = add(sum, scale(L, 1.0f / numSamples));
    }
    return sum;
}

// PathTrace, render.cpp:230-388
vec3 path_trace(const tb200_scene& sc, vec3 origin, vec3 dir, float time, int maxDepth, rng_t& rng)
{
    vec3 T = splat(1.0f), total = splat(0.0f);
    vec3 ro = origin, rd = dir;
    float rayEta = 1.0f;
    vec3 rayAbs = splat(0.0f);
    int rayType = REFLECTED;
    float bsdfPdf = 1.0f;
    for (int i = 0; i < maxDepth; ++i) {
        hit_t h = closest_hit(sc, ro, rd, time);
        if (h.prim >= 0) {
            COUNT(C_HIT, 1);
            const tb200_primitive& prim = sc.primitives[h.prim];
            float outEta;
            vec3 outAbs;
            if (rayEta == 1.0f) {
                outEta = mat_ior(prim.material);
                outAbs = from(prim.material.absorption);
            } else {
                outEta = 1.0f;
                outAbs = splat(0.0f);
            }
            vec3 e = scale(neg(rayAbs), h.t);
            T = mul(T, mk(tbm_expf(e.x), tbm_expf(e.y), tbm_expf(e.z)));
            vec3 p = add(ro, scale(rd, h.t));
            vec3 n = h.n;
            vec3 emission = from(prim.material.emission);
            if (i == 0) {
                total = add(total, emission);
            } else {
                float area = prim_area(sc, prim);
                if (area > 0.0f) {
                    float lightPdf = ((1.0f / area) * h.t * h.t) / clampf(dot3(neg(rd), n), 1.e-3f, 1.0f);
                    int N = int(prim.lightSamples + 1.0f);
                    float cbsdf = 1.0f / N, clight = float(prim.lightSamples) / N;
                    float weight = cbsdf * bsdfPdf / (cbsdf * bsdfPdf + clight * lightPdf);
                    if (rayType == SPECULAR) weight = 1.0f;
                    total = add(total, mul(scale(T, weight), emission));
                }
            }
            total = add(total, mul(T, sample_lights(sc, prim, rayEta, outEta, p, n, neg(rd), time, rng)));
            if (prim.lightSamples) break;
            vec3 u, v;
            basis(n, u, v);
            vec3 bdir = splat(0.0f);
            int btype = REFLECTED;
            bsdf_sample(prim.material, rayEta, outEta, u, v, n, neg(rd), bdir, bsdfPdf, btype, rng);
            if (bsdfPdf <= 0.0f) break;
            vec3 f = bsdf_eval(prim.material, rayEta, outEta, n, neg(rd), bdir);
            if (dot3(bdir, n) <= 0.0f) {
                rayEta = outEta;
                rayAbs = outAbs;
            }
            T = mul(T, divs(scale(f, absf(dot3(n, bdir))), bsdfPdf));
            rayType = btype;
            rd = bdir;
            ro = add(p, scale(face_fwd(n, bdir), RAY_EPS));
        } else {
            COUNT(C_MISS_BYTES, sc.sky.probeValid ? 16 : 0);
            float weight = 1.0f;
            if (sc.sky.probeValid && i > 0 && rayType != SPECULAR) {
                COUNT(C_MISS_BYTES, 8);
                float skyPdf = probe_pdf(sc.sky, rd);
                float cbsdf = 1.0f / 2, csky = 1.0f / 2;
                weight = cbsdf * bsdfPdf / (cbsdf * bsdfPdf + csky * skyPdf);
            }
            total = add(total, mul(scale(sky_eval(sc.sky, rd), weight), T));
            break;
        }
    }
    return total;
}

// ---- camera + film, util.h:45-83, render.cpp:401-445 -----------------------------------------------

struct camera_t {
    float r2w[4][4];   // [col][row]
    vec3 origin;
};

void mat4_mul(const float a[4][4], const float b[4][4], float out[4][4])   // MatrixMultiply<4,4,4>, maths.h:86-101
{
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j) {
            float t = 0.0f;
            for (int k = 0; k < 4; ++k) t += a[k][i] * b[j][k];
            out[j][i] = t;
        }
}

camera_t make_camera(const tb200_camera& c, int width, int height)   // CameraSampler ctor, util.h:49-71
{
    quat q{c.rotation[0], c.rotation[1], c.rotation[2], c.rotation[3]};
    float s = 1.0f;
    vec3 c0 = scale(qrot(q, mk(1, 0, 0)), s), c1 = scale(qrot(q, mk(0, 1, 0)), s), c2 = scale(qrot(q, mk(0, 0, 1)), s);
    vec3 c3 = scale(from(c.position), s);
    float c2w[4][4] = {{c0.x, c0.y, c0.z, 0.0f}, {c1.x, c1.y, c1.z, 0.0f}, {c2.x, c2.y, c2.z, 0.0f}, {c3.x, c3.y, c3.z, 1.0f}};
    float r2s[4][4] = {{2.0f / width, 0, 0, 0}, {0, -2.0f / height, 0, 0}, {0, 0, 1.0f, 0}, {-1.0f, 1.0f, 1.0f, 1.0f}};
    float f = tanf(c.fov * 0.5f);
    float aspect = float(width) / height;
    float s2c[4][4] = {{f * aspect, 0, 0, 0}, {0, f, 0, 0}, {0, 0, -1.0f, 0}, {0, 0, 0, 1.0f}};
    float tmp[4][4];
    camera_t cam;
    mat4_mul(c2w, s2c, tmp);
    mat4_mul(tmp, r2s, cam.r2w);
    cam.origin = mk(c2w[3][0], c2w[3][1], c2w[3][2]);
    return cam;
}

void generate_ray(const camera_t& cam, float rx, float ry, vec3& origin, vec3& dir)   // util.h:73-79, maths.h:923-930
{
    const float(*m)[4] = cam.r2w;
    vec3 p;
    p.x = m[0][0] * rx + m[1][0] * ry + m[2][0] * 0.0f + m[3][0];
    p.y = m[0][1] * rx + m[1][1] * ry + m[2][1] * 0.0f + m[3][1];
    p.z = m[0][2] * rx + m[1][2] * ry + m[2][2] * 0.0f + m[3][2];
    origin = cam.origin;
    dir = unit(sub(p, origin));
}

float filter_gauss(const tb200_options& o, float x) { return fmax2(0.0f, tbm_expf(-o.filterFalloff * x * x) - o.filterOffset); }   // render.h:29-32

void add_sample(const tb200_options& o, float* out, int W, int H, float rx, float ry, vec3 sample)   // render.cpp:401-445
{
    int sx = imax2(0, int(rx - o.filterWidth)), sy = imax2(0, int(ry - o.filterWidth));
    int ex = imin2(int(rx + o.filterWidth), W - 1), ey = imin2(int(ry + o.filterWidth), H - 1);
    vec3 c = sample;
    float l = len3(sample);
    if (l > o.clamp) c = scale(sample, o.clamp / l);   // ClampLength, maths.h:1577-1589
    COUNT(C_SAMPLES, 1);
    for (int x = sx; x <= ex; ++x)
        for (int y = sy; y <= ey; ++y) {
            COUNT(C_FB_PIXELS, 1);
            float w = 1.0f;
            float* px = out + 4 * ((size_t)y * W + x);
            if (o.filterType == TB200_FILTER_GAUSSIAN) {
                w = filter_gauss(o, x - rx) * filter_gauss(o, y - ry);
                px[0] += c.x * w; px[1] += c.y * w; px[2] += c.z * w; px[3] += w;
            } else {
                px[0] += c.x; px[1] += c.y; px[2] += c.z; px[3] += 1.0f;
            }
        }
}

struct sample_t {
    float rx, ry;
    vec3 radiance;
};

// one iteration of the raster loop, render.cpp:470-490, with a per-(pixel,frame) seed
sample_t trace_sample(const tb200_scene& sc, const tb200_camera& cam, const camera_t& cs, const tb200_options& o, int i, int j, int frame)
{
    rng_t rng = rng_make(tb200_sample_seed((uint32_t)(j * o.width + i), (uint32_t)frame));
    float x = rng_f(rng), y = rng_f(rng);
    float t = rng_f(rng);
    float time = mixf(cam.shutterStart, cam.shutterEnd, t);
    x += i;
    y += j;
    vec3 origin, dir;
    generate_ray(cs, x, y, origin, dir);
    sample_t s;
    s.rx = x;
    s.ry = y;
    s.radiance = path_trace(sc, origin, dir, time, o.maxDepth, rng);
    return s;
}

template <typename F>
void parallel_bands(int H, int nthreads, F body)
{
    if (nthreads < 1) nthreads = 1;
    if (nthreads > H) nthreads = H;
    std::vector<std::thread> th;
    for (int t = 0; t < nthreads; ++t) {
        int r0 = int((long long)H * t / nthreads), r1 = int((long long)H * (t + 1) / nthreads);
        th.emplace_back(body, t, r0, r1);
    }
    for (auto& x : th) x.join();
}

}  // namespace

extern "C" {

void* oracle_create(const tb200_scene* scene) { return new Oracle{scene}; }

// work counters since the last reset (all zero unless built with -DTB_ORACLE_COUNT)
int oracle_counters(unsigned long long* out, int reset)
{
#ifdef TB_ORACLE_COUNT
    for (int i = 0; i < C_NUM; ++i) {
        out[i] = g_counters[i].load();
        if (reset) g_counters[i].store(0);
    }
    return C_NUM;
#else
    for (int i = 0; i < C_NUM; ++i) out[i] = 0;
    (void)reset;
    return 0;
#endif
}
void oracle_destroy(void* h) { delete (Oracle*)h; }

// Same contract as ref_render_seeded (oracle/ref_driver.cpp): adds frames into caller-zeroed sums.
void oracle_render_seeded(void* h, const tb200_camera* cam, const tb200_options* o, int frame0, int nframes, float* out, int nthreads)
{
    const tb200_scene& sc = *((Oracle*)h)->scene;
    const int W = o->width, H = o->height;
    const camera_t cs = make_camera(*cam, W, H);
    if (nthreads < 1) nthreads = 1;
    if (nthreads > H) nthreads = H;
    const int halo = int(o->filterWidth) + 1;
    std::vector<std::vector<float>> bufs(nthreads);
    parallel_bands(H, nthreads, [&](int tid, int r0, int r1) {
        const int b0 = imax2(0, r0 - halo), b1 = imin2(H, r1 + halo);
        bufs[tid].assign((size_t)W * (b1 - b0) * 4, 0.0f);
        float* base = bufs[tid].data() - (size_t)b0 * W * 4;
        for (int k = frame0; k < frame0 + nframes; ++k)
            for (int j = r0; j < r1; ++j)
                for (int i = 0; i < W; ++i) {
                    sample_t s = trace_sample(sc, *cam, cs, *o, i, j, k);
                    add_sample(*o, base, W, H, s.rx, s.ry, s.radiance);
                }
    });
    for (int t = 0; t < nthreads; ++t) {
        int r0 = int((long long)H * t / nthreads), r1 = int((long long)H * (t + 1) / nthreads);
        int b0 = imax2(0, r0 - halo), b1 = imin2(H, r1 + halo);
        for (int y = b0; y < b1; ++y)
            for (int x = 0; x < W * 4; ++x) out[(size_t)y * W * 4 + x] += bufs[t][(size_t)(y - b0) * W * 4 + x];
    }
}

void oracle_trace_frame(void* h, const tb200_camera* cam, const tb200_options* o, int frame, float* radiance, float* raster, int nthreads)
{
    const tb200_scene& sc = *((Oracle*)h)->scene;
    const int W = o->width, H = o->height;
    const camera_t cs = make_camera(*cam, W, H);
    parallel_bands(H, nthreads, [&](int, int r0, int r1) {
        for (int j = r0; j < r1; ++j)
            for (int i = 0; i < W; ++i) {
                sample_t s = trace_sample(sc, *cam, cs, *o, i, j, frame);
                size_t p = (size_t)j * W + i;
                radiance[p * 3 + 0] = s.radiance.x; radiance[p * 3 + 1] = s.radiance.y; radiance[p * 3 + 2] = s.radiance.z;
                raster[p * 2 + 0] = s.rx; raster[p * 2 + 1] = s.ry;
            }
    });
}

// eNormals, render.cpp:494-515
void oracle_render_normals(void* h, const tb200_camera* cam, const tb200_options* o, float* out)
{
    const tb200_scene& sc = *((Oracle*)h)->scene;
    const int W = o->width, H = o->height;
    const camera_t cs = make_camera(*cam, W, H);
    for (int j = 0; j < H; ++j)
        for (int i = 0; i < W; ++i) {
            vec3 origin, dir;
            generate_ray(cs, (float)i, (float)j, origin, dir);
            hit_t hit = closest_hit(sc, origin, dir, 1.0f);
            float* px = out + 4 * ((size_t)j * W + i);
            if (hit.prim >= 0) {
                vec3 n = add(scale(hit.n, 0.5f), splat(0.5f));
                px[0] = n.x; px[1] = n.y; px[2] = n.z; px[3] = 1.0f;
            } else {
                px[0] = px[1] = px[2] = px[3] = 0.0f;
            }
        }
}

// ---- known-answer hooks (same signatures as the ref_* hooks) ---------------------------------------
void oracle_random_u32(int seed, int n, uint32_t* out)
{
    rng_t r = rng_make((uint32_t)seed);
    for (int i = 0; i < n; ++i) out[i] = rng_u32(r);
}
void oracle_random_f32(int seed, int n, float* out)
{
    rng_t r = rng_make((uint32_t)seed);
    for (int i = 0; i < n; ++i) out[i] = rng_f(r);
}
float oracle_material_ior(const tb200_material* m) { return mat_ior(*m); }
void oracle_bsdf_eval(const tb200_material* m, float etaI, float etaO, const float* n, const float* v, const float* l, float* f, float* pdf)
{
    vec3 r = bsdf_eval(*m, etaI, etaO, from(n), from(v), from(l));
    f[0] = r.x; f[1] = r.y; f[2] = r.z;
    *pdf = bsdf_pdf(*m, etaI, etaO, from(n), from(v), from(l));
}
void oracle_bsdf_sample(const tb200_material* m, float etaI, float etaO, const float* n, const float* v, int seed, float* l, float* pdf,
                        int* type, uint32_t* rngAfter)
{
    vec3 U, W;
    basis(from(n), U, W);
    rng_t rng = rng_make((uint32_t)seed);
    vec3 L = splat(0.0f);
    float p = -1.0f;
    int t = REFLECTED;
    bsdf_sample(*m, etaI, etaO, U, W, from(n), from(v), L, p, t, rng);
    l[0] = L.x; l[1] = L.y; l[2] = L.z;
    *pdf = p;
    *type = t;
    rngAfter[0] = rng.a;
    rngAfter[1] = rng.b;
}
void oracle_generate_ray(const tb200_camera* c, int width, int height, float x, float y, float* origin, float* dir)
{
    camera_t cs = make_camera(*c, width, height);
    vec3 o, d;
    generate_ray(cs, x, y, o, d);
    origin[0] = o.x; origin[1] = o.y; origin[2] = o.z;
    dir[0] = d.x; dir[1] = d.y; dir[2] = d.z;
}
float oracle_filter_eval(int type, float width, float falloff, float offset, float x, float y)
{
    tb200_options o;
    memset(&o, 0, sizeof(o));
    o.filterType = type; o.filterWidth = width; o.filterFalloff = falloff; o.filterOffset = offset;
    if (type != TB200_FILTER_GAUSSIAN) return 1.0f;
    return filter_gauss(o, x) * filter_gauss(o, y);
}
int oracle_trace(void* h, const float* o, const float* d, float time, float* t, float* n)
{
    hit_t hit = closest_hit(*((Oracle*)h)->scene, from(o), from(d), time);
    *t = hit.t;
    n[0] = hit.n.x; n[1] = hit.n.y; n[2] = hit.n.z;
    return hit.prim;
}
void oracle_probe_sample(void* h, int seed, float* dir, float* color, float* pdf)
{
    rng_t rng = rng_make((uint32_t)seed);
    vec3 d, c;
    float p = 0.0f;
    probe_sample(((Oracle*)h)->scene->sky, d, c, p, rng);
    dir[0] = d.x; dir[1] = d.y; dir[2] = d.z;
    color[0] = c.x; color[1] = c.y; color[2] = c.z;
    *pdf = p;
}
void oracle_sky_eval(void* h, const float* d, float* color, float* pdf)
{
    const tb200_sky& s = ((Oracle*)h)->scene->sky;
    vec3 c = sky_eval(s, from(d));
    color[0] = c.x; color[1] = c.y; color[2] = c.z;
    *pdf = s.probeValid ? probe_pdf(s, from(d)) : 0.0f;
}
void oracle_primitive_sample(void* h, int prim, float time, int seed, float* pos, float* normal, float* area)
{
    const tb200_scene& sc = *((Oracle*)h)->scene;
    rng_t rng = rng_make((uint32_t)seed);
    vec3 p, n;
    prim_sample(sc, sc.primitives[prim], time, p, n, rng);
    pos[0] = p.x; pos[1] = p.y; pos[2] = p.z;
    normal[0] = n.x; normal[1] = n.y; normal[2] = n.z;
    *area = prim_area(sc, sc.primitives[prim]);
}

// ---- display/finish step (SURVEY 8f rank 1) ------------------------------------------------------
// src/main.cpp:262-271: s = exposure / w;  filtered = LinearToSrgb(ToneMap(pixel * s, limit)),
// ToneMap = filmic curve of util.h:25-42 then SrgbToLinear (maths.h:1551-1555), alpha 0.
static float finish_channel(float t)
{
    float b = t - 0.004f;
    float x = (0.0f < b) ? b : 0.0f;                           // Max(Vec3(0), c - Vec3(0.004)), maths.h:59
    float ret = (x * (6.2f * x + 0.5f)) / (x * (6.2f * x + 1.7f) + 0.06f);
    float lin = tbm_powf(ret, 2.2f);                           // SrgbToLinear, maths.h:1553-1554
    return tbm_powf(lin, 1.0f / 2.2f);                         // LinearToSrgb, maths.h:1547-1548
}
void oracle_finish(const float* pixels, int numPixels, float exposure, float limit, float* filtered)
{
    (void)limit;   // only the commented-out Reinhard branch of ToneMap reads it
    for (int i = 0; i < numPixels; ++i) {
        float s = exposure / pixels[i * 4 + 3];
        filtered[i * 4 + 0] = finish_channel(pixels[i * 4 + 0] * s);
        filtered[i * 4 + 1] = finish_channel(pixels[i * 4 + 1] * s);
        filtered[i * 4 + 2] = finish_channel(pixels[i * 4 + 2] * s);
        filtered[i * 4 + 3] = 0.0f;
    }
}
// src/png.cpp:324-343: the 8-bit buffer WritePng hands to TinyPngOut (one sequential Random(),
// two draws per channel; sum in double, narrowed to float, Clamp = Min(Max(x,0),255), truncated).
void oracle_quantize(const float* filtered, int numPixels, unsigned char* rgb8)
{
    rng_t rand = rng_make(0u);
    for (int i = 0; i < numPixels; ++i)
        for (int c = 0; c < 3; ++c) {
            float r1 = rng_f(rand);
            float r2 = rng_f(rand);
            float x = (float)((double)filtered[i * 4 + c] * 255.0 + (double)r1 + (double)r2 - (double)0.5f);
            x = (x < 0.0f) ? 0.0f : x;
            x = (x < 255.0f) ? x : 255.0f;
            rgb8[i * 3 + c] = (unsigned char)x;
        }
}

// ---- non-local means (SURVEY 8f rank 2), src/nlm.cpp ------------------------------------------------
// AverageFilter (nlm.cpp:4-34) then NonLocalMeansFilter (nlm.cpp:36-73): window clamped to the
// image, columns outer / rows inner, Color (4 floats) arithmetic, weight = expf(-falloff*LengthSq(dm)).
void oracle_nlm(const float* in, float* out, int width, int height, float falloff, int radius)
{
    std::vector<float> means((size_t)width * height * 4);
    for (int y = 0; y < height; ++y)
        for (int x = 0; x < width; ++x) {
            int xlower = std::max(0, x - radius), xupper = std::min(width - 1, x + radius);
            int ylower = std::max(0, y - radius), yupper = std::min(height - 1, y + radius);
            int count = 0;
            float sum[4] = {0.0f, 0.0f, 0.0f, 0.0f};
            for (int fx = xlower; fx <= xupper; ++fx)
                for (int fy = ylower; fy <= yupper; ++fy) {
                    const float* p = in + ((size_t)fy * width + fx) * 4;
                    for (int c = 0; c < 4; ++c) sum[c] = sum[c] + p[c];
                    count += 1;
                }
            float inv = 1.0f / count;
            for (int c = 0; c < 4; ++c) means[((size_t)y * width + x) * 4 + c] = sum[c] * inv;
        }
    for (int y = 0; y < height; ++y)
        for (int x = 0; x < width; ++x) {
            int xlower = std::max(0, x - radius), xupper = std::min(width - 1, x + radius);
            int ylower = std::max(0, y - radius), yupper = std::min(height - 1, y + radius);
            float totalWeight = 0.0f;
            float sum[4] = {0.0f, 0.0f, 0.0f, 0.0f};
            const float* mean = &means[((size_t)y * width + x) * 4];
            for (int fx = xlower; fx <= xupper; ++fx)
                for (int fy = ylower; fy <= yupper; ++fy) {
                    const float* m = &means[((size_t)fy * width + fx) * 4];
                    float dx = mean[0] - m[0], dy = mean[1] - m[1], dz = mean[2] - m[2], dw = mean[3] - m[3];
                    float weight = tbm_expf(-falloff * (dx * dx + dy * dy + dz * dz + dw * dw));
                    const float* p = in + ((size_t)fy * width + fx) * 4;
                    for (int c = 0; c < 4; ++c) sum[c] = sum[c] + p[c] * weight;
                    totalWeight += weight;
                }
            float inv = 1.0f / totalWeight;
            for (int c = 0; c < 4; ++c) out[((size_t)y * width + x) * 4 + c] = sum[c] * inv;
        }
}

}  // extern "C"
