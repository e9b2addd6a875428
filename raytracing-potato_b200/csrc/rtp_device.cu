// rtp_device.cu — sm_100a kernels and the device-facing half of the C ABI.
//
// Arithmetic contract: every expression below that restates a reference expression keeps the
// reference's association order, and this file is compiled with --fmad=false, so no multiply-add
// is contracted (rustc never fuses). f64 division and sqrt are IEEE-correct in CUDA. The only
// operations that may differ from the CPU by an ulp are atan2/asin (sphere and sky uv).
//
// Reference citations are file:line under /root/reference/src.

#include <cub/device/device_select.cuh>
#include <cuda_runtime.h>
#include <math_constants.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include "rtp_internal.h"

namespace rtp {

// A failed call also clears the runtime's last error, so that a refused call (an allocation that does not fit, say) does not
// fail the next call of this thread at its first cudaGetLastError(). A sticky error stays sticky: reading it changes nothing.
#define RTP_CUDA(expr)                                                                               \
    do {                                                                                             \
        cudaError_t _e = (expr);                                                                     \
        if (_e != cudaSuccess) {                                                                     \
            cudaGetLastError();                                                                      \
            return set_error(RTP_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));      \
        }                                                                                            \
    } while (0)

constexpr double kRayEpsilon = 1e-3;  // utility.rs:30
constexpr double kSmol = 1e-7;        // utility.rs:31
constexpr double kPi = 3.14159265358979323846264338327950288;
constexpr double kTau = 6.28318530717958647692528676655900577;

// ---------------------------------------------------------------------------------------------
// small device helpers
// ---------------------------------------------------------------------------------------------

struct D3 {
    double x, y, z;
};
__device__ __forceinline__ D3 mk(double x, double y, double z) { return D3{x, y, z}; }
__device__ __forceinline__ D3 operator-(D3 a, D3 b) { return mk(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ D3 operator+(D3 a, D3 b) { return mk(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ D3 operator*(double s, D3 a) { return mk(s * a.x, s * a.y, s * a.z); }
__device__ __forceinline__ D3 cmul(D3 a, D3 b) { return mk(a.x * b.x, a.y * b.y, a.z * b.z); }
// nalgebra 0.29 reductions on static 3-vectors
__device__ __forceinline__ double dot(D3 a, D3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
__device__ __forceinline__ double norm_squared(D3 a) { return 0.0 + dot(a, a); }
__device__ __forceinline__ double norm(D3 a) { return sqrt(norm_squared(a)); }
__device__ __forceinline__ D3 normalize(D3 a) {
    const double n = norm(a);
    return mk(a.x / n, a.y / n, a.z / n);
}

__device__ __forceinline__ double2 ldg2(const double* p) { return __ldg(reinterpret_cast<const double2*>(p)); }

struct Counters {
    unsigned long long rays, paths, node_visits, triangle_tests, sphere_tests, leaf_gates, violations, rewalks;
    // lane occupancy of trace_any_kernel's rounds (counting builds, RTP_LANE_STATS=1 prints them): per round, how many lanes could
    // walk, sat on two pending leaves, had a leaf pending but nothing left to walk, or held no ray
    unsigned long long rounds, lanes_walk, lanes_full, lanes_leafwait, lanes_empty, leaf_rounds, leaf_lanes, step_lanes;
};

struct LocalCounters {
    unsigned int rays, node_visits, triangle_tests, sphere_tests, leaf_gates, violations, rewalks;
};

// ---------------------------------------------------------------------------------------------
// K1: closest hit. Restates bvh.rs:93-124 as a stack-free pre-order walk (see rtp_internal.h).
// ---------------------------------------------------------------------------------------------

struct HitRec {
    double t;       // in: ray.t_max, out: t of the closest hit (unchanged on miss)
    double u, v;    // triangle barycentrics of the winner
    uint32_t slot;  // primitive slot of the winner, kNoPrim on miss
    uint32_t kind;  // rtp_hittable_kind of the winner
};

// utility.rs:137-154 AABB::collide — literal form (12 minNum/maxNum)
__device__ __forceinline__ bool collide_literal(const double2 b0, const double2 b1, const double2 b2, D3 o, D3 inv, double ray_tmin,
                                                double ray_tmax) {
    // b0 = (min.x, min.y), b1 = (min.z, max.x), b2 = (max.y, max.z)
    const double t0x = (b0.x - o.x) * inv.x, t0y = (b0.y - o.y) * inv.y, t0z = (b1.x - o.z) * inv.z;
    const double t1x = (b1.y - o.x) * inv.x, t1y = (b2.x - o.y) * inv.y, t1z = (b2.y - o.z) * inv.z;
    const double t_min = fmax(fmax(fmax(ray_tmin, fmin(t0x, t1x)), fmin(t0y, t1y)), fmin(t0z, t1z));
    const double t_max = fmin(fmin(fmin(ray_tmax, fmax(t0x, t1x)), fmax(t0y, t1y)), fmax(t0z, t1z));
    return t_max >= t_min;
}

// Same decision as collide_literal for rays whose origin is finite, whose 1/direction is finite and non-zero on all
// three axes, and whose t_min <= t_max are not NaN (no NaN can then appear in any lane):
//   * IEEE rounding is monotone, so for inv > 0: (min-o)*inv <= (max-o)*inv and min(t0,t1) is the min-plane value; for
//     inv < 0 it is the max-plane value. Picking the plane by the sign of inv replaces the six inner min/max, and
//     far_a >= near_a holds on every axis.
//   * without NaNs, min(T,fx,fy,fz) >= max(tmin,nx,ny,nz) is the conjunction of the pairwise comparisons; the four that
//     are always true (T >= tmin is kept true by the caller, far_a >= near_a) are dropped, leaving twelve.
// No value is selected, so the decision is a pure predicate chain. Other rays use collide_literal.
__device__ __forceinline__ bool collide_fast(const double2 b0, const double2 b1, const double2 b2, D3 o, D3 inv, bool sx, bool sy, bool sz,
                                             double tmin, double T) {
    const double pnx = sx ? b1.y : b0.x, pfx = sx ? b0.x : b1.y;
    const double pny = sy ? b2.x : b0.y, pfy = sy ? b0.y : b2.x;
    const double pnz = sz ? b2.y : b1.x, pfz = sz ? b1.x : b2.y;
    const double nx = (pnx - o.x) * inv.x, ny = (pny - o.y) * inv.y, nz = (pnz - o.z) * inv.z;
    const double fx = (pfx - o.x) * inv.x, fy = (pfy - o.y) * inv.y, fz = (pfz - o.z) * inv.z;
    const bool p0 = (T >= nx) & (T >= ny) & (T >= nz);
    const bool p1 = (fx >= tmin) & (fx >= ny) & (fx >= nz);
    const bool p2 = (fy >= tmin) & (fy >= nx) & (fy >= nz);
    const bool p3 = (fz >= tmin) & (fz >= nx) & (fz >= ny);
    return p0 & p1 & p2 & p3;
}

// Conservative f32 culling. Inputs: a child's outward-inflated f32 box (rtp_internal.h DWide), inv32 = RN32(1/d), and per
// axis c_lo = RD32(-(o*inv) - K), c_hi = RU32(-(o*inv) + K) with K = 2^-21 |o*inv| + 1e-37. Then
//   n_lo = fma(near_plane, inv32, c_lo) <= the f64 slab entry (min-o)*inv as the reference rounds it, and
//   f_hi = fma(far_plane,  inv32, c_hi) >= the f64 slab exit,
// for |o|, |box| <= 1e15 and 1e-15 <= |inv| <= 1e15 (no overflow/underflow trouble); the derivation is in DESIGN.md §4.
// With T_up >= t_max and tmin_dn <= t_min, `min(T_up, f_hi) < max(tmin_dn, n_lo)` therefore implies that the reference's
// f64 test `t_max >= t_min` is false for this box and for every box inside it: the subtree can be skipped. The converse
// is not claimed: a child that is not rejected here is simply visited, and leaves get the exact f64 gate.
struct Ray32 {
    float ix, iy, iz;
    float clx, cly, clz, chx, chy, chz;
    float tmin_dn, T_up;
};

// the four children of one DWide node at once: bit k of the result = child k is NOT rejected
__device__ __forceinline__ uint32_t collide32_wide(const float4 nx4, const float4 fx4, const float4 ny4, const float4 fy4, const float4 nz4,
                                                   const float4 fz4, const Ray32& r) {
#define RTP_CHILD(c)                                                                                                        \
    (fminf(fminf(fmaf(fx4.c, r.ix, r.chx), fmaf(fy4.c, r.iy, r.chy)), fminf(fmaf(fz4.c, r.iz, r.chz), r.T_up)) >=          \
     fmaxf(fmaxf(fmaf(nx4.c, r.ix, r.clx), fmaf(ny4.c, r.iy, r.cly)), fmaxf(fmaf(nz4.c, r.iz, r.clz), r.tmin_dn)))
    // `>=` on finite-or-infinite operands is exactly !(tf < tn); no NaN can occur for an f32-eligible ray (finite inv, finite
    // or infinite planes of one sign per product)
    return (RTP_CHILD(x) ? 1u : 0u) | (RTP_CHILD(y) ? 2u : 0u) | (RTP_CHILD(z) ? 4u : 0u) | (RTP_CHILD(w) ? 8u : 0u);
#undef RTP_CHILD
}

__device__ __forceinline__ bool in_f32_range(double x) { const double a = fabs(x); return a >= 1e-15 && a <= 1e15; }

__device__ __forceinline__ bool finite_nonzero(double x) { return x != 0.0 && fabs(x) <= 1.7976931348623157e308; }
__device__ __forceinline__ bool finite(double x) { return fabs(x) <= 1.7976931348623157e308; }

// hittable.rs:65-108 hit_triangle up to the accept test
__device__ __forceinline__ bool test_triangle(const DPrim* __restrict__ p, D3 o, D3 d, double ray_tmin, double ray_tmax, double& t_out,
                                              double& u_out, double& v_out) {
    const double* pd = reinterpret_cast<const double*>(p);  // a[3] ba[3] ca[3] are contiguous
    const double2 q0 = ldg2(pd), q1 = ldg2(pd + 2), q2 = ldg2(pd + 4), q3 = ldg2(pd + 6);
    const double q4 = __ldg(pd + 8);
    const D3 a = mk(q0.x, q0.y, q1.x);
    const D3 ba = mk(q1.y, q2.x, q2.y);
    const D3 ca = mk(q3.x, q3.y, q4);
    const D3 pa = a - o;

    const double det = ba.x * ca.y * d.z + ba.y * ca.z * d.x + ba.z * ca.x * d.y - ba.x * ca.z * d.y - ba.y * ca.x * d.z -
                       ba.z * ca.y * d.x;
    if (fabs(det) < kSmol) return false;
    const double inv_det = 1.0 / det;

    const double t = (pa.x * (ba.y * ca.z - ba.z * ca.y) + pa.y * (ba.z * ca.x - ba.x * ca.z) + pa.z * (ba.x * ca.y - ba.y * ca.x)) * inv_det;
    const double u = (pa.x * (ca.y * d.z - ca.z * d.y) + pa.y * (ca.z * d.x - ca.x * d.z) + pa.z * (ca.x * d.y - ca.y * d.x)) * inv_det;
    const double v = (pa.x * (ba.z * d.y - ba.y * d.z) + pa.y * (ba.x * d.z - ba.z * d.x) + pa.z * (ba.y * d.x - ba.x * d.y)) * inv_det;
    const double w = 1.0 - u - v;
    if (t < ray_tmin || t > ray_tmax || u < 0.0 || v < 0.0 || w < 0.0) return false;
    t_out = t; u_out = u; v_out = v;
    return true;
}

// hittable.rs:39-57 hit_sphere up to the accepted root
__device__ __forceinline__ bool test_sphere(const DPrim* __restrict__ p, D3 o, D3 d, double ray_tmin, double ray_tmax, double& t_out) {
    const double* pd = reinterpret_cast<const double*>(p);  // center in a[], radius in ba[0]
    const double2 q0 = ldg2(pd), q1 = ldg2(pd + 2);
    const D3 center = mk(q0.x, q0.y, q1.x);
    const double radius = q1.y;
    const D3 to_center = o - center;
    const double a = norm_squared(d);
    const double half_b = dot(d, to_center);
    const double c = norm_squared(to_center) - radius * radius;
    const double delta = half_b * half_b - a * c;
    if (delta <= 0.0) return false;
    const double sqrt_delta = sqrt(delta);
    double t = (-half_b - sqrt_delta) / a;
    if (t < ray_tmin || t > ray_tmax) {
        t = (-half_b + sqrt_delta) / a;
        if (t < ray_tmin || t > ray_tmax) return false;
    }
    t_out = t;
    return true;
}

// bvh.rs:121-124 Bvh::hit. `h.t` carries ray.t_max in and the closest t out.
template <bool COUNT>
__device__ __forceinline__ void closest_hit_bvh(const DSceneView& sc, D3 o, D3 d, double ray_tmin, HitRec& h, LocalCounters& lc) {
    const D3 inv = mk(1.0 / d.x, 1.0 / d.y, 1.0 / d.z);  // utility.rs:71-77 Ray::expand
    const DNode* __restrict__ nodes = sc.nodes;
    const uint32_t n_nodes = sc.n_nodes;
    uint32_t node = 0;
    h.slot = kNoPrim;
    for (;;) {
        // walk until a leaf passes its own slab gate (bvh.rs:96, 103) or the tree is exhausted
        uint32_t prim = kNoPrim, kind = 0;
        while (node < n_nodes) {
            const double* nb = nodes[node].bmin;
            const double2 b0 = ldg2(nb), b1 = ldg2(nb + 2), b2 = ldg2(nb + 4);
            const uint4 meta = __ldg(reinterpret_cast<const uint4*>(nb + 6));
            if (COUNT) lc.node_visits++;
            if (collide_literal(b0, b1, b2, o, inv, ray_tmin, h.t)) {
                node = node + 1;
                if (meta.y != kNoPrim) { prim = meta.y; kind = meta.z; break; }
            } else {
                node = meta.x;
            }
        }
        if (prim == kNoPrim) break;
        const DPrim* p = sc.prims + prim;
        double t, u = 0.0, v = 0.0;
        bool hit;
        if (kind == RTP_HITTABLE_TRIANGLE) {
            if (COUNT) lc.triangle_tests++;
            hit = test_triangle(p, o, d, ray_tmin, h.t, t, u, v);
        } else {
            if (COUNT) lc.sphere_tests++;
            hit = test_sphere(p, o, d, ray_tmin, h.t, t);
        }
        if (hit) {  // bvh.rs:107-111: shrink t_max, later hit replaces
            h.t = t; h.u = u; h.v = v; h.slot = prim; h.kind = kind;
        }
    }
}

// hittable.rs:110-120 hit_list over the primitive list in caller order
template <bool COUNT>
__device__ __forceinline__ void closest_hit_list(const DSceneView& sc, D3 o, D3 d, double ray_tmin, HitRec& h, LocalCounters& lc) {
    h.slot = kNoPrim;
    const D3 inv = mk(1.0 / d.x, 1.0 / d.y, 1.0 / d.z);  // only read for gated items (leaves of a nested Bvh, bvh.rs:121-124)
    for (uint32_t slot = 0; slot < sc.n_prims; ++slot) {
        const uint2 kp = __ldg(reinterpret_cast<const uint2*>(&sc.nodes[slot].kind));  // kind, gate flag
        const uint32_t kind = kp.x;
        const DPrim* p = sc.prims + slot;
        if (kp.y) {  // bvh.rs:96: the leaf's own box first
            const double* pb = p->bmin;
            if (COUNT) lc.leaf_gates++;
            if (!collide_literal(ldg2(pb), ldg2(pb + 2), ldg2(pb + 4), o, inv, ray_tmin, h.t)) continue;
        }
        double t, u = 0.0, v = 0.0;
        bool hit;
        if (kind == RTP_HITTABLE_TRIANGLE) {
            if (COUNT) lc.triangle_tests++;
            hit = test_triangle(p, o, d, ray_tmin, h.t, t, u, v);
        } else {
            if (COUNT) lc.sphere_tests++;
            hit = test_sphere(p, o, d, ray_tmin, h.t, t);
        }
        if (hit) { h.t = t; h.u = u; h.v = v; h.slot = slot; h.kind = kind; }
    }
}

template <bool COUNT>
__device__ __forceinline__ void closest_hit(const DSceneView& sc, D3 o, D3 d, double ray_tmin, HitRec& h, LocalCounters& lc) {
    lc.rays++;
    if (sc.root_kind == RTP_ROOT_BVH) closest_hit_bvh<COUNT>(sc, o, d, ray_tmin, h, lc);
    else closest_hit_list<COUNT>(sc, o, d, ray_tmin, h, lc);
}

// The rest of `Hit` for the winner (hittable.rs:58-62, 102-107). Pure function of (ray, t, u, v,
// primitive), so evaluating it once after traversal gives the bits the reference computed at accept time.
struct Surface {
    D3 position, normal;
    double u, v;
    uint32_t material, leaf;
};

__device__ __forceinline__ void finish_hit(const DSceneView& sc, D3 o, D3 d, const HitRec& h, Surface& s) {
    const DPrim* p = sc.prims + h.slot;
    s.leaf = __ldg(&p->leaf);
    s.material = __ldg(&p->material);
    s.position = o + h.t * d;  // utility.rs:67-69 Ray::at
}

__device__ __forceinline__ void finish_triangle(const DSceneView& sc, const HitRec& h, Surface& s) {
    const DAttr* at = sc.attrs + h.slot;
    const double w = 1.0 - h.u - h.v;
    const double* n = &at->n[0][0];
    const double2 a0 = ldg2(n), a1 = ldg2(n + 2), a2 = ldg2(n + 4), a3 = ldg2(n + 6);
    const double a4 = __ldg(n + 8);
    const D3 n0 = mk(a0.x, a0.y, a1.x), n1 = mk(a1.y, a2.x, a2.y), n2 = mk(a3.x, a3.y, a4);
    s.normal = (w * n0 + h.u * n1) + h.v * n2;  // hittable.rs:105, not renormalised
    const double* uv = &at->uv[0][0];
    const double2 u0 = ldg2(uv), u1 = ldg2(uv + 2), u2 = ldg2(uv + 4);
    s.u = (w * u0.x + h.u * u1.x) + h.v * u2.x;  // hittable.rs:106
    s.v = (w * u0.y + h.u * u1.y) + h.v * u2.y;
}

__device__ __forceinline__ void finish_sphere(const DSceneView& sc, const HitRec& h, Surface& s, bool want_uv = true) {
    const DPrim* p = sc.prims + h.slot;
    const double* pd = reinterpret_cast<const double*>(p);
    const double2 q0 = ldg2(pd), q1 = ldg2(pd + 2);
    const D3 center = mk(q0.x, q0.y, q1.x);
    s.normal = normalize(s.position - center);  // hittable.rs:60
    if (want_uv) {
        s.u = 0.5 - atan2(s.normal.z, s.normal.x) / kTau;  // hittable.rs:61
        s.v = asin(s.normal.y) / kPi + 0.5;
    } else {
        s.u = 0.0; s.v = 0.0;  // never read: see material_reads_uv
    }
}

// Hit::uv (hittable.rs:61) is only consumed by Texture::sample (texture.rs:21-36), i.e. by an AlbedoMap absorb or a
// SkySphere emit of the hit material; the two f64 transcendentals of the sphere uv are skipped for every other material.
__device__ __forceinline__ bool material_reads_uv(const DMaterial* m) {
    return __ldg(&m->absorb) == RTP_ABSORB_ALBEDO_MAP || __ldg(&m->emit_kind) == RTP_EMIT_SKY_SPHERE;
}

// ---------------------------------------------------------------------------------------------
// kernels: ray batches
// ---------------------------------------------------------------------------------------------

// Output record of the traversal kernel inside the wavefront integrator: what shading needs to rebuild the
// reference's `Hit` (t, barycentrics, primitive slot | kind << 31; slot == kNoPrim on a miss). 32 bytes.
struct alignas(16) WaveHit {
    double t, u, v;
    uint32_t slotkind, _pad;
};
static_assert(sizeof(WaveHit) == 32, "WaveHit must be 32 bytes");

// OUT_OCCLUDED: one byte per ray, 1 iff the ray hits anything (the in-order kernel stops at the first accepted leaf, DESIGN.md §2c)
enum { OUT_HIT = 0, OUT_FULL = 1, OUT_WAVE = 2, OUT_TAIL = 3, OUT_OCCLUDED = 4 };

template <int OUT>
__device__ __forceinline__ void write_hit(const DSceneView& sc, void* __restrict__ out, size_t i, D3 o, D3 d, const HitRec& h) {
    if (OUT == OUT_FULL) {
        rtp_hit_full* o_full = static_cast<rtp_hit_full*>(out) + i;
        rtp_hit_full r;
        if (h.slot != kNoPrim) {
            Surface s;
            finish_hit(sc, o, d, h, s);
            if (h.kind == RTP_HITTABLE_TRIANGLE) finish_triangle(sc, h, s);
            else finish_sphere(sc, h, s);
            r.leaf = s.leaf; r.material = s.material; r.t = h.t;
            r.position[0] = s.position.x; r.position[1] = s.position.y; r.position[2] = s.position.z;
            r.normal[0] = s.normal.x; r.normal[1] = s.normal.y; r.normal[2] = s.normal.z;
            r.uv[0] = s.u; r.uv[1] = s.v;
        } else {
            memset(&r, 0, sizeof r);
            r.leaf = RTP_MISS; r.material = RTP_MISS; r.t = CUDART_INF;
        }
        *o_full = r;
    } else if (OUT == OUT_WAVE) {
        double2* w = reinterpret_cast<double2*>(static_cast<WaveHit*>(out) + i);
        w[0] = make_double2(h.t, h.u);
        w[1] = make_double2(h.v, __hiloint2double(0, static_cast<int>(h.slot == kNoPrim ? kNoPrim : (h.slot | (h.kind << 31)))));
    } else if (OUT == OUT_OCCLUDED) {
        static_cast<uint8_t*>(out)[i] = h.slot != kNoPrim ? 1u : 0u;
    } else {
        uint4 w;
        if (h.slot != kNoPrim) {
            const DPrim* p = sc.prims + h.slot;
            w.x = __ldg(&p->leaf); w.y = __ldg(&p->material);
            const unsigned long long tb = static_cast<unsigned long long>(__double_as_longlong(h.t));
            w.z = static_cast<uint32_t>(tb); w.w = static_cast<uint32_t>(tb >> 32);
        } else {
            w.x = RTP_MISS; w.y = RTP_MISS;
            w.z = 0u; w.w = 0x7FF00000u;  // +inf
        }
        reinterpret_cast<uint4*>(out)[i] = w;
    }
}

// one atomic per warp per counter
template <bool COUNT>
__device__ __forceinline__ void flush_counters(Counters* counters, const LocalCounters& lc) {
    if (!counters) return;
    unsigned int r = lc.rays, nv = lc.node_visits, tt = lc.triangle_tests, st = lc.sphere_tests, lg = lc.leaf_gates, vi = lc.violations, rw = lc.rewalks;
    for (int off = 16; off; off >>= 1) {
        r += __shfl_down_sync(0xffffffffu, r, off);
        if (COUNT) {
            nv += __shfl_down_sync(0xffffffffu, nv, off);
            tt += __shfl_down_sync(0xffffffffu, tt, off);
            st += __shfl_down_sync(0xffffffffu, st, off);
            lg += __shfl_down_sync(0xffffffffu, lg, off);
            vi += __shfl_down_sync(0xffffffffu, vi, off);
            rw += __shfl_down_sync(0xffffffffu, rw, off);
        }
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&counters->rays, static_cast<unsigned long long>(r));
        if (COUNT) {
            atomicAdd(&counters->node_visits, static_cast<unsigned long long>(nv));
            atomicAdd(&counters->triangle_tests, static_cast<unsigned long long>(tt));
            atomicAdd(&counters->sphere_tests, static_cast<unsigned long long>(st));
            atomicAdd(&counters->leaf_gates, static_cast<unsigned long long>(lg));
            atomicAdd(&counters->violations, static_cast<unsigned long long>(vi));
            if (rw) atomicAdd(&counters->rewalks, static_cast<unsigned long long>(rw));
        }
    }
}

// Baseline kernels: one thread per ray, no regrouping. Kept for A/B runs (RTP_TRACE_KERNEL=simple).
template <bool COUNT, int OUT>
__device__ __forceinline__ void trace_closest_one(const DSceneView& sc, const rtp_ray* __restrict__ rays, size_t n, void* __restrict__ out,
                                                  Counters* counters) {
    const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    LocalCounters lc = {0, 0, 0, 0, 0, 0, 0};
    if (i < n) {
        const double2* rp = reinterpret_cast<const double2*>(rays + i);
        const double2 r0 = __ldg(rp), r1 = __ldg(rp + 1), r2 = __ldg(rp + 2), r3 = __ldg(rp + 3);
        const D3 o = mk(r0.x, r0.y, r1.x), d = mk(r1.y, r2.x, r2.y);
        HitRec h;
        h.t = r3.y; h.u = 0.0; h.v = 0.0; h.kind = 0;
        closest_hit<COUNT>(sc, o, d, r3.x, h, lc);
        write_hit<OUT>(sc, out, i, o, d, h);
    }
    flush_counters<COUNT>(counters, lc);
}

template <bool COUNT, bool FULL>
__global__ void __launch_bounds__(128) trace_closest_kernel(DSceneView sc, const rtp_ray* __restrict__ rays, size_t n, void* __restrict__ out,
                                                            Counters* counters) {
    trace_closest_one<COUNT, FULL ? OUT_FULL : OUT_HIT>(sc, rays, n, out, counters);
}

// occlusion: the closest hit, then `slot != kNoPrim`, which is the definition of the answer itself
template <bool COUNT>
__global__ void __launch_bounds__(128) trace_occluded_simple_kernel(DSceneView sc, const rtp_ray* __restrict__ rays, size_t n, void* __restrict__ out,
                                                                    Counters* counters) {
    trace_closest_one<COUNT, OUT_OCCLUDED>(sc, rays, n, out, counters);
}

// ---------------------------------------------------------------------------------------------
// Persistent wavefront traversal. One warp owns 32 ray slots and keeps them busy:
//   * lanes whose ray has finished pull new ray indices from a global counter (one atomic per
//     refill, ranks by ballot), so a warp never idles behind its longest ray;
//   * lanes that reach a leaf whose slab gate passes park until enough lanes are parked, then
//     the primitive tests run together (ballot-batched), so the expensive triangle/sphere code
//     is not executed for one lane at a time.
// Every lane still performs exactly the reference's sequence of tests for its ray (pre-order
// walk, bvh.rs:93-119), so results are independent of how rays are grouped.
// ---------------------------------------------------------------------------------------------

struct WorkQueue {
    unsigned long long next;   // next unclaimed ray index
    unsigned int done_blocks;  // warps that have drained; the last one resets the queue for the next launch
    unsigned int _pad;
};

// Rays the pure any-order kernel (trace_any_kernel) does not answer itself: not eligible for the f32 walk, stack overflow, or an
// abnormal leaf inside the final window. The in-order kernel traces them in a second launch (its `index` mode).
struct DeferList {
    uint32_t* idx;               // ray indices handed to the in-order kernel
    unsigned long long* count;   // entries in idx (device); reset by the in-order launch that consumes it
};

// Thresholds of both persistent kernels (measured: DESIGN.md §6)
constexpr int kRefillMin = 16;  // refill when at least this many lanes are empty
constexpr int kPrimBatch = 4;   // run primitive tests when at least this many lanes are parked at a leaf
constexpr int kMinLanes = 1;    // smallest number of rays a warp holds when the batch is small

// Per-lane traversal state.
//   f32-eligible lanes (m32) walk the 4-wide culling tree: `next` = node to visit, (cur, pend, c0..c3) = node whose
//   children are being handed out, pending-children mask and its child words; a short stack of (node << 4 | mask)
//   entries in shared memory holds the ancestors that still have pending children.
//   Other lanes (non-finite or axis-parallel rays, huge coordinates, List roots) walk the exact f64 pre-order tree with
//   `next` as the pre-order index (bvh.rs:93-119 literally).
constexpr uint32_t kEnd = 0xFFFFFFFFu;   // `next`: the walk is over
constexpr uint32_t kNone = 0xFFFFFFFEu;  // `next`: no node to visit, take the next pending child
struct Walker {
    D3 o, d, inv;
    double tmin;
    HitRec h;        // h.t is the running t_max
    Ray32 r32;
    uint32_t next;
    uint32_t cur, pend, sp;
    uint32_t c0, c1, c2, c3;
    uint32_t onx, ony, onz;  // byte offset of the near plane inside each axis block of a DWide (0 or 16)
    uint32_t prim;   // kNoPrim, or slot | kind << 31 of the oldest leaf handed out and not tested yet
    uint32_t prim2;  // f32 walk only: a second pending leaf. The lane keeps walking (with a stale, larger t_max: conservative)
                     // until two leaves are pending; they are tested strictly in the order they were handed out
    bool fast;       // eligible for collide_fast (finite, non-axis-parallel, no NaN)
    bool m32;        // eligible for the f32 culling walk
    bool need_gate;  // parked by the f32 walk: the leaf's exact f64 gate has not been evaluated yet
    bool sx, sy, sz;
};

// utility.rs:71-77 Ray::expand plus the derived quantities of the fast paths
__device__ __forceinline__ void walker_start(Walker& w, const DSceneView& sc, D3 o, D3 d, double tmin, double tmax) {
    w.o = o; w.d = d;
    w.inv = mk(1.0 / d.x, 1.0 / d.y, 1.0 / d.z);
    w.tmin = tmin;
    w.h.t = tmax; w.h.u = 0.0; w.h.v = 0.0; w.h.slot = kNoPrim; w.h.kind = 0;
    w.fast = sc.fast_slab && finite_nonzero(w.inv.x) && finite_nonzero(w.inv.y) && finite_nonzero(w.inv.z) && finite(o.x) && finite(o.y) &&
             finite(o.z) && tmax >= tmin;
    w.sx = w.inv.x < 0.0; w.sy = w.inv.y < 0.0; w.sz = w.inv.z < 0.0;
    w.m32 = w.fast && sc.f32_culling && in_f32_range(w.inv.x) && in_f32_range(w.inv.y) && in_f32_range(w.inv.z) &&
            fabs(o.x) <= 1e15 && fabs(o.y) <= 1e15 && fabs(o.z) <= 1e15;
    if (w.m32) {
        const double px = o.x * w.inv.x, py = o.y * w.inv.y, pz = o.z * w.inv.z;
        const double kx = fabs(px) * 0x1.0p-21 + 1e-37, ky = fabs(py) * 0x1.0p-21 + 1e-37, kz = fabs(pz) * 0x1.0p-21 + 1e-37;
        w.r32.ix = __double2float_rn(w.inv.x); w.r32.iy = __double2float_rn(w.inv.y); w.r32.iz = __double2float_rn(w.inv.z);
        w.r32.clx = __double2float_rd(-px - kx); w.r32.cly = __double2float_rd(-py - ky); w.r32.clz = __double2float_rd(-pz - kz);
        w.r32.chx = __double2float_ru(-px + kx); w.r32.chy = __double2float_ru(-py + ky); w.r32.chz = __double2float_ru(-pz + kz);
        w.r32.tmin_dn = __double2float_rd(tmin);
        w.r32.T_up = __double2float_ru(tmax);
        w.onx = w.sx ? 16u : 0u; w.ony = w.sy ? 16u : 0u; w.onz = w.sz ? 16u : 0u;
    }
    w.next = 0;
    w.pend = 0; w.sp = 0; w.cur = 0;
    w.prim = kNoPrim; w.prim2 = kNoPrim;
    w.need_gate = false;
}

// One step of an f32-eligible lane that is walking (next != kEnd, not parked): visit `next` if there is one (four
// conservative slab tests), then hand out the next pending child in rank order: a leaf parks the lane, an internal
// child becomes `next`. `stack` is this thread's column of the shared-memory stack (stride = blockDim.x).
template <bool COUNT>
__device__ __forceinline__ void walker_step_wide(Walker& w, const DSceneView& sc, LocalCounters& lc, uint32_t* __restrict__ stack, uint32_t stride) {
    if (w.next != kNone) {
        const char* np = reinterpret_cast<const char*>(sc.wide + w.next);
        const float4 nx4 = __ldg(reinterpret_cast<const float4*>(np + w.onx));
        const float4 fx4 = __ldg(reinterpret_cast<const float4*>(np + (16u - w.onx)));
        const float4 ny4 = __ldg(reinterpret_cast<const float4*>(np + 32u + w.ony));
        const float4 fy4 = __ldg(reinterpret_cast<const float4*>(np + 32u + (16u - w.ony)));
        const float4 nz4 = __ldg(reinterpret_cast<const float4*>(np + 64u + w.onz));
        const float4 fz4 = __ldg(reinterpret_cast<const float4*>(np + 64u + (16u - w.onz)));
        const uint4 ch = __ldg(reinterpret_cast<const uint4*>(np + 96u));
        w.pend = collide32_wide(nx4, fx4, ny4, fy4, nz4, fz4, w.r32);
        if (COUNT) {
            lc.node_visits++;
            const double* b64 = sc.wide_boxes + static_cast<size_t>(w.next) * 24;
            for (uint32_t k = 0; k < 4; ++k)  // the conservative test must never reject a box the exact test accepts
                if (!((w.pend >> k) & 1u) && (&ch.x)[k] != kWideEmpty &&
                    collide_literal(ldg2(b64 + 6 * k), ldg2(b64 + 6 * k + 2), ldg2(b64 + 6 * k + 4), w.o, w.inv, w.tmin, w.h.t))
                    lc.violations++;
        }
        w.c0 = ch.x; w.c1 = ch.y; w.c2 = ch.z; w.c3 = ch.w;
        w.cur = w.next;
        w.next = kNone;
    }
    if (w.pend == 0u) {
        if (w.sp == 0u) { w.next = kEnd; return; }
        w.sp -= 1u;
        const uint32_t e = stack[w.sp * stride];
        w.cur = e >> 4; w.pend = e & 15u;
        const uint4 ch = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const char*>(sc.wide + w.cur) + 96u));
        w.c0 = ch.x; w.c1 = ch.y; w.c2 = ch.z; w.c3 = ch.w;
    }
    // hand out the lowest pending child; everything below is selects and one predicated store, no branches
    const uint32_t k = __ffs(w.pend) - 1u;
    w.pend &= w.pend - 1u;
    const uint32_t s1 = (k & 1u) << 5;  // clamped funnel shifts pick one of four 32-bit words
    const uint32_t c = __funnelshift_rc(__funnelshift_rc(w.c0, w.c1, s1), __funnelshift_rc(w.c2, w.c3, s1), (k & 2u) << 4);
    const bool is_leaf = (c & kWideLeaf) != 0u;
    const uint32_t leaf = ((c >> 30) & 1u) << 31 | (c & kWideSlotMask);
    const bool first = w.prim == kNoPrim;
    w.prim2 = (is_leaf & !first) ? leaf : w.prim2;
    w.prim = (is_leaf & first) ? leaf : w.prim;
    w.need_gate = w.need_gate | is_leaf;
    const bool push = !is_leaf & (w.pend != 0u);
    if (push) stack[w.sp * stride] = (w.cur << 4) | w.pend;
    w.sp += push ? 1u : 0u;
    w.next = is_leaf ? kNone : c;
}

// ---------------------------------------------------------------------------------------------
// Any-order walk (DESIGN.md §4b): trace_any_kernel, further down. The reference's result is that of the sequential process
//     T = ray.t_max; for leaf p in DFS order: if T >= m_p: T = t_p, best = p
// where, for a leaf that passes its static tests (box entered at all, barycentrics inside, t_p >= t_min), t_p is the computed
// hit distance and m_p = max(t_p, computed slab entry of p's own box) — both independent of T. A leaf is NORMAL when
// m_p = t_p and ABNORMAL when rounding put t_p below its own box entry. If every leaf with t_p <= M + 2 slack is normal, where
// M is the smallest m_p, the process returns min t_p, ties to the larger DFS rank — no matter in which order the leaves are
// looked at. slack(t) bounds m_p - t_p for every primitive that is not "big" (error analysis of hittable.rs:39-57, 77-95 in
// DESIGN.md §4b), so a box whose conservative entry lies above T_win = t_best + 2 slack(t_best) holds no leaf that can matter and
// is skipped, children are visited nearest first, and the primitive tests use T_win as their upper bound. Big primitives (the
// outsized ones of a scene, at most eight) are tested for every ray before its walk starts. A ray that met an abnormal leaf inside
// the final window is traced again in the reference's order by the kernel below (its index mode): exactness never rests on the
// bound being tight, only on it being a bound.
// ---------------------------------------------------------------------------------------------

// One exact f64 step for lanes outside the f32 path's preconditions (bvh.rs:93-119 literally, or collide_fast).
template <bool COUNT>
__device__ __forceinline__ void walker_step64(Walker& w, const DSceneView& sc, LocalCounters& lc) {
    const double* nb = sc.nodes[w.next].bmin;
    const double2 b0 = ldg2(nb), b1 = ldg2(nb + 2), b2 = ldg2(nb + 4);
    const uint4 meta = __ldg(reinterpret_cast<const uint4*>(nb + 6));
    if (COUNT) lc.node_visits++;
    const bool pass = w.fast ? collide_fast(b0, b1, b2, w.o, w.inv, w.sx, w.sy, w.sz, w.tmin, w.h.t) : collide_literal(b0, b1, b2, w.o, w.inv, w.tmin, w.h.t);
    w.next = pass ? w.next + 1 : meta.x;
    if (w.next >= sc.n_nodes) w.next = kEnd;
    if (pass & (meta.y != kNoPrim)) { w.prim = meta.y | (meta.z << 31); w.need_gate = false; }
}

// The parked lane's leaf: exact slab gate (bvh.rs:96) if still owed, then the primitive (bvh.rs:97), then un-park.
template <bool COUNT>
__device__ __forceinline__ void walker_leaf(Walker& w, const DSceneView& sc, LocalCounters& lc) {
    const uint32_t slot = w.prim & 0x7FFFFFFFu, kind = w.prim >> 31;
    const DPrim* p = sc.prims + slot;
    // bvh.rs:96-97 accepts a leaf iff its slab gate AND its primitive test pass; both are pure functions of (ray, t_max,
    // leaf), so the order of evaluation is free. The gate passes for ~94% of the leaves the f32 walk hands out, so the
    // primitive goes first and the exact gate only confirms an accepted hit. The counting kernels keep the reference's
    // order, so their test counters are the oracle's.
    bool open = true;
    if (COUNT && w.need_gate) {
        const double* pb = p->bmin;
        lc.leaf_gates++;
        open = collide_fast(ldg2(pb), ldg2(pb + 2), ldg2(pb + 4), w.o, w.inv, w.sx, w.sy, w.sz, w.tmin, w.h.t);
    }
    if (open) {
        double t, u = 0.0, v = 0.0;
        bool hit;
        if (kind == RTP_HITTABLE_TRIANGLE) {
            if (COUNT) lc.triangle_tests++;
            hit = test_triangle(p, w.o, w.d, w.tmin, w.h.t, t, u, v);
        } else {
            if (COUNT) lc.sphere_tests++;
            hit = test_sphere(p, w.o, w.d, w.tmin, w.h.t, t);
        }
        if (!COUNT && hit && w.need_gate) {
            const double* pb = p->bmin;
            hit = collide_fast(ldg2(pb), ldg2(pb + 2), ldg2(pb + 4), w.o, w.inv, w.sx, w.sy, w.sz, w.tmin, w.h.t);
        }
        if (hit) {  // bvh.rs:107-111: shrink t_max, later hit replaces
            w.h.t = t; w.h.u = u; w.h.v = v; w.h.slot = slot; w.h.kind = kind;
            w.r32.T_up = __double2float_ru(t);
            // NaN t: only with overflowing (> 1e150) geometry, which the f32 walk's preconditions (|coordinates| <= 1e15) exclude;
            // a lane of the exact walk drops back to the literal slab test, whose NaN rules are the reference's
            if (!(t == t)) w.fast = false;
        }
    }
    w.prim = w.prim2;
    w.prim2 = kNoPrim;
}

// ---------------------------------------------------------------------------------------------
// camera (render.rs:32-52) — tan(fov/2) is evaluated on the host (glibc, like the reference's
// f64::tan) and passed in, so no device transcendental sits on the primary-ray path.
// ---------------------------------------------------------------------------------------------

struct DCamera {
    double tan_fov, focal_dist, aspect_ratio, lens_radius;
    double m[9];  // orientation, columns x, y, z
    double pos[3];
};

__device__ __forceinline__ void camera_shoot(const DCamera& cam, double u, double v, double lens_x, double lens_y, D3& o, D3& d) {
    const D3 origin = mk(lens_x, lens_y, 0.0);
    const D3 target = mk((2.0 * u - 1.0) * cam.tan_fov * cam.focal_dist * cam.aspect_ratio, (2.0 * v - 1.0) * cam.tan_fov * cam.focal_dist,
                         -cam.focal_dist);
    const D3 dir = normalize(target - origin);
    const double* m = cam.m;
    // utility.rs:185-191: orientation * v accumulates column by column
    d = mk((m[0] * dir.x + m[3] * dir.y) + m[6] * dir.z, (m[1] * dir.x + m[4] * dir.y) + m[7] * dir.z,
           (m[2] * dir.x + m[5] * dir.y) + m[8] * dir.z);
    o = mk(((m[0] * origin.x + m[3] * origin.y) + m[6] * origin.z) + cam.pos[0], ((m[1] * origin.x + m[4] * origin.y) + m[7] * origin.z) + cam.pos[1],
           ((m[2] * origin.x + m[5] * origin.y) + m[8] * origin.z) + cam.pos[2]);
}

// a ray from o along d with the reference's interval [kRayEpsilon, inf) (render.rs:104)
__device__ __forceinline__ void store_ray(rtp_ray* r, D3 o, D3 d) {
    double2* out = reinterpret_cast<double2*>(r);
    out[0] = make_double2(o.x, o.y);
    out[1] = make_double2(o.z, d.x);
    out[2] = make_double2(d.y, d.z);
    out[3] = make_double2(kRayEpsilon, CUDART_INF);
}

// writes the rays of pixels [first, first + count) (i fastest) to rays[0 .. count)
__global__ void __launch_bounds__(256) camera_rays_kernel(DCamera cam, uint32_t width, uint32_t height, rtp_ray* __restrict__ rays_out, size_t first, size_t count) {
    const size_t q = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (q >= count) return;
    const size_t p = first + q;
    rtp_ray* rays = rays_out - first;
    const uint32_t i = static_cast<uint32_t>(p % width), j = static_cast<uint32_t>(p / width);
    const double u = (static_cast<double>(i) + 0.5) / static_cast<double>(width);
    const double v = (static_cast<double>(j) + 0.5) / static_cast<double>(height);
    D3 o, d;
    camera_shoot(cam, u, v, 0.0, 0.0, o, d);
    store_ray(rays + p, o, d);
}

// ---------------------------------------------------------------------------------------------
// random stream (replaces StdRng; layout in rtp.h)
// ---------------------------------------------------------------------------------------------

struct Rng {
    uint32_t k0, k1, c0, c1, c3;
    uint32_t k;       // next draw
    uint32_t cached;  // block held in b0..b3
    uint32_t b0, b1, b2, b3;
};

__device__ __forceinline__ void rng_init(Rng& r, unsigned long long seed, uint32_t lo, uint32_t hi, uint32_t stream) {
    r.k0 = static_cast<uint32_t>(seed); r.k1 = static_cast<uint32_t>(seed >> 32);
    r.c0 = lo; r.c1 = hi; r.c3 = stream;
    r.k = 0; r.cached = 0xFFFFFFFFu;
    r.b0 = r.b1 = r.b2 = r.b3 = 0;
}

__device__ __forceinline__ void philox_block(Rng& r, uint32_t block) {
    uint32_t c0 = r.c0, c1 = r.c1, c2 = block, c3 = r.c3, k0 = r.k0, k1 = r.k1;
#pragma unroll
    for (int round = 0; round < 10; ++round) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    r.b0 = c0; r.b1 = c1; r.b2 = c2; r.b3 = c3;
    r.cached = block;
}

// rng.gen::<f64>() with rand 0.8's Standard mapping: 53 high bits * 2^-53
__device__ __forceinline__ double rng_next(Rng& r) {
    const uint32_t block = r.k >> 1, pair = r.k & 1u;
    if (block != r.cached) philox_block(r, block);
    r.k++;
    const uint32_t lo = pair ? r.b2 : r.b0, hi = pair ? r.b3 : r.b1;
    const unsigned long long u = (static_cast<unsigned long long>(hi) << 32) | lo;
    return static_cast<double>(u >> 11) * 0x1.0p-53;
}

// randomness.rs:21-34 / 39-53 / 58-73
__device__ __forceinline__ void sample_unit_disk(Rng& r, double& x, double& y) {
    for (;;) {
        const double vx = 2.0 * rng_next(r) - 1.0;
        const double vy = 2.0 * rng_next(r) - 1.0;
        if (0.0 + (vx * vx + vy * vy) < 1.0) { x = vx; y = vy; return; }
    }
}
__device__ __forceinline__ D3 sample_unit_ball(Rng& r) {
    for (;;) {
        D3 v;
        v.x = 2.0 * rng_next(r) - 1.0;
        v.y = 2.0 * rng_next(r) - 1.0;
        v.z = 2.0 * rng_next(r) - 1.0;
        if (norm_squared(v) < 1.0) return v;
    }
}
__device__ __forceinline__ D3 sample_unit_sphere(Rng& r) {
    for (;;) {
        const double vx = 2.0 * rng_next(r) - 1.0;
        const double vy = 2.0 * rng_next(r) - 1.0;
        const double s = 0.0 + (vx * vx + vy * vy);
        if (s < 1.0) {
            const double n = 2.0 * sqrt(1.0 - s);
            return mk(vx * n, vy * n, 1.0 - 2.0 * s);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// textures (texture.rs) and materials (material.rs)
// ---------------------------------------------------------------------------------------------

// Rust `as u32` / `as isize`: saturating, NaN -> 0
// cvt.rzi saturates like Rust, but maps NaN to 0x80000000 / INT64_MIN where Rust's `as` gives 0
__device__ __forceinline__ uint32_t sat_u32(double x) { return x != x ? 0u : __double2uint_rz(x); }
__device__ __forceinline__ long long sat_i64(double x) { return x != x ? 0ll : __double2ll_rz(x); }
// f64::clamp: NaN stays NaN
__device__ __forceinline__ double clampd(double x, double lo, double hi) { return x < lo ? lo : (x > hi ? hi : x); }

// randomness.rs:91-110
__device__ __forceinline__ long long noise_integer(long long x, long long y, long long z, long long seed) {
    const unsigned long long A = 0x369E6D3B899E43CFull, B = 0x53F89E7FFDA3B07Dull, C = 0x3B13C1CA4937E629ull, D = 0x577C2C6E4019D645ull;
    unsigned long long h = A * static_cast<unsigned long long>(x) + B * static_cast<unsigned long long>(y) + C * static_cast<unsigned long long>(z) +
                           D * static_cast<unsigned long long>(seed);
    h = static_cast<unsigned long long>(static_cast<long long>(h) >> 13) ^ h;
    h = h * (h * h * 60493ull + 19990303ull) + 1376312589ull;
    return static_cast<long long>(h);
}
__device__ __forceinline__ double noise_real(long long x, long long y, long long z, long long seed) {
    return static_cast<double>(noise_integer(x, y, z, seed)) / 9223372036854775808.0;
}
__device__ __forceinline__ double grad_dot(D3 p, long long cx, long long cy, long long cz, long long seed) {  // texture.rs:70-76
    const D3 g = mk(noise_real(cx, cy, cz, seed + 1), noise_real(cx, cy, cz, seed + 2), noise_real(cx, cy, cz, seed + 3));
    return dot(p - mk(static_cast<double>(cx), static_cast<double>(cy), static_cast<double>(cz)), g);
}
__device__ __forceinline__ double mixd(double a, double b, double t) { return (b - a) * t + a; }
__device__ __forceinline__ double smootherstep(double t) { return (t * (t * 6.0 - 15.0) + 10.0) * t * t * t; }

// texture.rs:20-36 Texture::sample. Checker recursion (texture.rs:51-60) is unrolled into a bounded loop;
// the reference would overflow its stack on a cyclic checker, here 64 hops yield black.
__device__ D3 texture_sample(const DSceneView& sc, uint32_t tid, D3 position, double hu, double hv) {
    for (int hop = 0; hop < 64; ++hop) {
        const DTexture* tx = sc.textures + tid;
        const uint32_t kind = __ldg(&tx->kind);
        switch (kind) {
            case RTP_TEXTURE_MISSING: return mk(0.0, 0.0, 0.0);
            case RTP_TEXTURE_DEBUG_UVS: return mk(hu, hv, 0.0);
            case RTP_TEXTURE_SOLID: return mk(__ldg(&tx->rgb[0]), __ldg(&tx->rgb[1]), __ldg(&tx->rgb[2]));
            case RTP_TEXTURE_IMAGE: {  // texture.rs:40-49
                const uint32_t wi = __ldg(&tx->width), hi = __ldg(&tx->height);
                const double w = static_cast<double>(wi), h = static_cast<double>(hi);
                const uint32_t i = sat_u32(clampd(hu * w, 0.0, w - 1.0));
                const uint32_t j = sat_u32(clampd(hv * h, 0.0, h - 1.0));
#ifdef RTP_DEVICE_CHECKS
                if (i >= wi || j >= hi || tid >= 64) printf("texture_sample: tid %u i %u j %u of %u x %u (hu %g hv %g)\n", tid, i, j, wi, hi, hu, hv);
#endif
                const uchar4* texels = reinterpret_cast<const uchar4*>(tx->rgba);
                const uchar4 px = __ldg(texels + (static_cast<size_t>(i) + static_cast<size_t>(j) * wi));  // image.rs:31-33
                return mk(static_cast<double>(px.x) / 255.0, static_cast<double>(px.y) / 255.0, static_cast<double>(px.z) / 255.0);
            }
            case RTP_TEXTURE_CHECKER: {
                const double sum = floor(position.x) + floor(position.y) + floor(position.z);
                tid = (fmod(sum, 2.0) == 0.0) ? __ldg(&tx->even) : __ldg(&tx->odd);
                continue;
            }
            case RTP_TEXTURE_NOISE: {  // texture.rs:62-68
                double x = noise_real(sat_i64(floor(position.x)), sat_i64(floor(position.y)), sat_i64(floor(position.z)), tx->seed);
                x = 0.5 * x + 0.5;
                return mk(x, x, x);
            }
            case RTP_TEXTURE_PERLIN: {  // texture.rs:82-119
                const D3 p = position;
                const D3 fp = mk(floor(p.x), floor(p.y), floor(p.z));
                const long long flx = sat_i64(fp.x), fly = sat_i64(fp.y), flz = sat_i64(fp.z);
                const long long clx = flx + 1, cly = fly + 1, clz = flz + 1;
                const long long seed = tx->seed;
                const double k1 = grad_dot(p, flx, fly, flz, seed), k2 = grad_dot(p, clx, fly, flz, seed);
                const double k3 = grad_dot(p, flx, cly, flz, seed), k4 = grad_dot(p, clx, cly, flz, seed);
                const double k5 = grad_dot(p, flx, fly, clz, seed), k6 = grad_dot(p, clx, fly, clz, seed);
                const double k7 = grad_dot(p, flx, cly, clz, seed), k8 = grad_dot(p, clx, cly, clz, seed);
                D3 t = p - fp;
                t = mk(smootherstep(t.x), smootherstep(t.y), smootherstep(t.z));
                const double k12 = mixd(k1, k2, t.x), k34 = mixd(k3, k4, t.x), k56 = mixd(k5, k6, t.x), k78 = mixd(k7, k8, t.x);
                const double k1234 = mixd(k12, k34, t.y), k5678 = mixd(k56, k78, t.y);
                const double x = 0.5 * mixd(k1234, k5678, t.z) + 0.5;
                return mk(x, x, x);
            }
            default: return mk(0.0, 0.0, 0.0);
        }
    }
    return mk(0.0, 0.0, 0.0);
}

// material.rs:49-60 Emit::evaluate
__device__ __forceinline__ D3 emit_evaluate(const DSceneView& sc, uint32_t kind, uint32_t tex, const double* rgb, D3 dir, D3 position, D3 normal,
                                            double hu, double hv) {
    switch (kind) {
        case RTP_EMIT_COLOR: return mk(rgb[0], rgb[1], rgb[2]);
        case RTP_EMIT_DEBUG_NORMALS: return normal;
        case RTP_EMIT_SKY_GRADIENT: {
            const double t = 0.5 * (dir.y / norm(dir) + 1.0);
            const double a = 1.0 - t;
            return mk(a * 1.0 + t * 0.5, a * 1.0 + t * 0.7, a * 1.0 + t * 1.0);
        }
        case RTP_EMIT_SKY_SPHERE: return texture_sample(sc, tex, position, hu, hv);
        default: return mk(0.0, 0.0, 0.0);
    }
}

// utility.rs:106-108
__device__ __forceinline__ D3 reflect(D3 incident, D3 normal) { return incident - (2.0 * dot(incident, normal)) * normal; }

// ---------------------------------------------------------------------------------------------
// K2-K6: the per-pixel bounce loop (main.rs:70-83 + render.rs:94-146).
//
// One path vertex is shaded by shade_vertex(): it rebuilds the reference's `Hit` for the winner,
// runs Material::evaluate (scatter -> absorb -> emit, material.rs:104-110) and either ends the path
// or produces the scattered ray. Radiance is folded inside-out like the recursion (render.rs:108-115):
// (emit, absorb) of every scattering vertex go on a per-path stack and are combined when the path ends.
// Per-sample colours go to a scratch buffer and are summed in sample order by resolve_kernel, which
// reproduces the reference's sequential `final_color += ...` (main.rs:80) bit for bit.
// ---------------------------------------------------------------------------------------------

struct DRender {
    uint32_t width, height, max_bounce;
    uint32_t tile_x, tile_y, tile_w, tile_h;
    uint32_t sample_begin;  // first sample of this launch
    uint32_t n_samples;     // samples per pixel in this launch
    uint32_t row_offset;    // this launch covers rows tile_y + row_offset + k * row_stride, k < tile_h (rtp_render_params.row_*:
    uint32_t row_stride;    //   a frame split by rows over devices or processes); tile_h counts the rows of THIS launch
    uint32_t _pad;
    unsigned long long seed;
};

// Which tile pixel the k-th pixel slot of a launch is, as a compile-time policy of the integrator kernels. A launch has
// map.count(rp) slots; the tile pixel index is row-major over the rows of this launch (rp.tile_w wide).
struct DenseTile {  // rtp_render: every pixel of the tile rectangle, slot k = tile pixel k
    __device__ __forceinline__ size_t count(const DRender& rp) const { return static_cast<size_t>(rp.tile_w) * rp.tile_h; }
    __device__ __forceinline__ uint32_t pixel(uint32_t k) const { return k; }
};
struct LiveList {   // rtp_render_adaptive: the pixels still sampling in this round, slot k = tile pixel live[k]
    const uint32_t* live;
    uint32_t n;
    __device__ __forceinline__ size_t count(const DRender&) const { return n; }
    __device__ __forceinline__ uint32_t pixel(uint32_t k) const { return __ldg(live + k); }
};

// What a path's first vertex leaves for rtp_render_aov (DESIGN.md §6c): the material's absorb there and Hit::normal; (0, 0, 0) on a miss
struct FirstVertex {
    D3 albedo, normal;
};

// Whether the integrator kernels capture each path's FirstVertex, as a compile-time policy. A launch with AovRecords writes one
// 48-byte record per path p: (albedo.x, albedo.y) (albedo.z, normal.x) (normal.y, normal.z) at rec + 3 p.
struct NoAov {  // rtp_render, rtp_render_srgb8, rtp_render_adaptive
    static constexpr bool kOn = false;
    __device__ __forceinline__ void record(size_t, const FirstVertex&) const {}
};
struct AovRecords {  // rtp_render_aov
    static constexpr bool kOn = true;
    double2* rec;
    __device__ __forceinline__ void record(size_t p, const FirstVertex& f) const {
        double2* r = rec + 3 * p;
        r[0] = make_double2(f.albedo.x, f.albedo.y);
        r[1] = make_double2(f.albedo.z, f.normal.x);
        r[2] = make_double2(f.normal.y, f.normal.z);
    }
};

// path p of a launch = (pixel slot p / n_samples, sample p % n_samples): the samples of one pixel sit in adjacent lanes,
// so a warp's primary rays are as coherent as they can be. Returns the path's random stream at its first draw; (i, j) is its
// frame pixel.
template <class Map>
__device__ __forceinline__ Rng path_rng(const DRender& rp, const Map& map, size_t p, uint32_t& i, uint32_t& j) {
    // a launch holds at most 32 Mi paths (render_enqueue): 32-bit divisions (the 64-bit ones were 3.6 % of the shade kernel)
    const uint32_t p32 = static_cast<uint32_t>(p);
    const uint32_t k = p32 / rp.n_samples;
    const uint32_t smp = rp.sample_begin + (p32 - k * rp.n_samples);
    const uint32_t pix = map.pixel(k);
    const uint32_t row = pix / rp.tile_w;
    i = rp.tile_x + (pix - row * rp.tile_w);
    j = rp.tile_y + rp.row_offset + row * rp.row_stride;
    Rng rng;
    rng_init(rng, rp.seed, j * rp.width + i, smp, RTP_RNG_STREAM_PATH);
    return rng;
}

// main.rs:70-76: jittered uv (render.rs:76-81), lens sample (render.rs:36, drawn even when lens_radius == 0), Camera::shoot
__device__ __forceinline__ void primary_ray(const DCamera& cam, const DRender& rp, uint32_t i, uint32_t j, Rng& rng, D3& o, D3& d) {
    const double u = (static_cast<double>(i) + rng_next(rng)) / static_cast<double>(rp.width);
    const double v = (static_cast<double>(j) + rng_next(rng)) / static_cast<double>(rp.height);
    double lx, ly;
    sample_unit_disk(rng, lx, ly);
    camera_shoot(cam, u, v, cam.lens_radius * lx, cam.lens_radius * ly, o, d);
}

// render.rs:118,144 + utility.rs:93-100 Hit::at_infinity + background.evaluate
__device__ __forceinline__ D3 shade_miss(const DSceneView& sc, D3 d) {
    const double hu = 0.5 - atan2(d.z, d.x) / kTau, hv = asin(d.y) / kPi + 0.5;
    return emit_evaluate(sc, sc.bg_kind, sc.bg_texture, sc.bg_rgb, d, d, d, hu, hv);
}

// render.rs:105-115 for a hit: returns true when the material scattered (then o, d hold the scattered ray, render.rs:111-114).
// fv != nullptr: the vertex's absorb and Hit::normal are stored there too (rtp_render_aov's first vertex).
__device__ __forceinline__ bool shade_vertex(const DSceneView& sc, D3& o, D3& d, const HitRec& h, Rng& rng, D3& emit, D3& absorb,
                                             FirstVertex* fv = nullptr) {
    Surface s;
#ifdef RTP_DEVICE_CHECKS
    if (h.slot >= sc.n_prims) printf("shade_vertex: slot %u of %u kind %u t %g\n", h.slot, sc.n_prims, h.kind, h.t);
#endif
    finish_hit(sc, o, d, h, s);
#ifdef RTP_DEVICE_CHECKS
    if (s.material >= 64) printf("shade_vertex: material %u slot %u\n", s.material, h.slot);
#endif
    const DMaterial* m = sc.materials + s.material;
    if (h.kind == RTP_HITTABLE_TRIANGLE) finish_triangle(sc, h, s);
    else finish_sphere(sc, h, s, material_reads_uv(m));
    // every scattering material draws at least once: generate the block of the next draw here, where all lanes of the warp
    // are still together, instead of inside the per-material branches (the stream itself is unchanged)
    if (__ldg(&m->scatter) != RTP_SCATTER_NONE) philox_block(rng, rng.k >> 1);

    // material.rs:104-110: scatter, then absorb, then emit
    bool scattered = false;
    D3 sd = mk(0.0, 0.0, 0.0);
    const uint32_t scatter = __ldg(&m->scatter);
    if (scatter == RTP_SCATTER_LAMBERT) {  // material.rs:115-130
        if (!(dot(s.normal, d) > 0.0)) {
            sd = normalize(s.normal + sample_unit_sphere(rng));
            scattered = true;
        }
    } else if (scatter == RTP_SCATTER_METAL) {  // material.rs:132-152
        if (!(dot(s.normal, d) > 0.0)) {
            const D3 refl = reflect(d, s.normal);
            const D3 fz = __ldg(&m->scatter_param) * sample_unit_ball(rng);
            sd = normalize(refl + fz);
            scattered = !(dot(s.normal, sd) < 0.0);
        }
    } else if (scatter == RTP_SCATTER_DIELECTRIC) {  // material.rs:154-180
        const double ior = __ldg(&m->scatter_param);
        double eta;
        D3 n;
        if (dot(s.normal, d) > 0.0) { eta = ior; n = mk(-s.normal.x, -s.normal.y, -s.normal.z); }
        else { eta = 1.0 / ior; n = s.normal; }
        const double q = (1.0 - eta) / (1.0 + eta);
        const double r0 = q * q;  // powi(2)
        const double x = 1.0 + dot(n, d);
        const double x2 = x * x;
        const double reflectance = r0 + (1.0 - r0) * (x * (x2 * x2));  // powi(5)
        if (rng_next(rng) < reflectance) {
            sd = reflect(d, n);
        } else {  // utility.rs:110-119 refract, else reflect
            const double cos_theta = dot(n, d);
            const double k = 1.0 - eta * eta * (1.0 - cos_theta * cos_theta);
            if (k < 0.0) sd = reflect(d, n);
            else sd = eta * d - (eta * cos_theta + sqrt(k)) * n;
        }
        scattered = true;
    }
    switch (__ldg(&m->absorb)) {  // material.rs:74-81
        case RTP_ABSORB_WHITEBODY: absorb = mk(1.0, 1.0, 1.0); break;
        case RTP_ABSORB_ALBEDO: absorb = mk(__ldg(&m->absorb_rgb[0]), __ldg(&m->absorb_rgb[1]), __ldg(&m->absorb_rgb[2])); break;
        case RTP_ABSORB_ALBEDO_MAP: absorb = texture_sample(sc, __ldg(&m->absorb_texture), s.position, s.u, s.v); break;
        default: absorb = mk(0.0, 0.0, 0.0); break;
    }
    emit = emit_evaluate(sc, __ldg(&m->emit_kind), __ldg(&m->emit_texture), m->emit_rgb, d, s.position, s.normal, s.u, s.v);
    if (fv) { fv->albedo = absorb; fv->normal = s.normal; }
    o = s.position; d = sd;
    return scattered;
}

// Baseline integrator: one thread per camera path, whole bounce loop in one thread, exact f64 stack-free walk.
// Kept for A/B runs (RTP_RENDER_KERNEL=simple) and as the second implementation the wavefront path is tested against.
template <int MAXB, bool COUNT, class Map, class Aov>
__global__ void __launch_bounds__(128) render_paths_kernel(DSceneView sc, DCamera cam, DRender rp, double4* __restrict__ scratch,
                                                            Counters* counters, Map map, Aov aov) {
    const size_t npix = map.count(rp);
    const size_t total = npix * rp.n_samples;
    const size_t p = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    LocalCounters lc = {0, 0, 0, 0, 0, 0, 0};
    if (p < total) {
        uint32_t i, j;
        Rng rng = path_rng(rp, map, p, i, j);
        D3 o, d;
        primary_ray(cam, rp, i, j, rng, o, d);

        double emit_stack[MAXB][3], absorb_stack[MAXB][3];
        int nb = 0;
        D3 L = mk(0.0, 0.0, 0.0);
        uint32_t depth = rp.max_bounce;
        bool first = true, first_hit = false;
        FirstVertex fv = {mk(0.0, 0.0, 0.0), mk(0.0, 0.0, 0.0)};
        for (;;) {
            if (!first && depth == 0) { L = mk(0.0, 0.0, 0.0); break; }  // render.rs:128-131
            HitRec h;
            h.t = CUDART_INF; h.u = 0.0; h.v = 0.0; h.kind = 0;
            closest_hit<COUNT>(sc, o, d, kRayEpsilon, h, lc);
            if (h.slot == kNoPrim) { L = shade_miss(sc, d); break; }
            if (first) first_hit = true;
            D3 emit, absorb;
            if (!shade_vertex(sc, o, d, h, rng, emit, absorb, Aov::kOn && first ? &fv : nullptr)) {  // render.rs:108-110: emit + rgb(0,0,0)
                L = emit + mk(0.0, 0.0, 0.0);
                break;
            }
            emit_stack[nb][0] = emit.x; emit_stack[nb][1] = emit.y; emit_stack[nb][2] = emit.z;
            absorb_stack[nb][0] = absorb.x; absorb_stack[nb][1] = absorb.y; absorb_stack[nb][2] = absorb.z;
            ++nb;
            depth -= 1;
            first = false;
        }
        // render.rs:108-115 / 135-142: emit + absorb ⊙ (inner), folded inside-out like the recursion
        for (int b = nb - 1; b >= 0; --b) {
            L = mk(emit_stack[b][0], emit_stack[b][1], emit_stack[b][2]) + cmul(mk(absorb_stack[b][0], absorb_stack[b][1], absorb_stack[b][2]), L);
        }
        scratch[p] = make_double4(L.x, L.y, L.z, first_hit ? 1.0 : 0.0);
        aov.record(p, fv);
    }
    flush_counters<COUNT>(counters, lc);
}

// ---------------------------------------------------------------------------------------------
// Wavefront integrator. A launch of P paths runs as
//     generate -> [ trace_persistent_kernel (OUT_WAVE) -> shade ] x max_bounce
// over ray queues in HBM. Queue b holds the rays of segment b of every path that is still alive, densely packed
// (shade compacts survivors with one atomic per warp), so the traversal kernel always sees full warps. Queue
// sizes live on the device (WaveQueues::count[b]); nothing synchronises with the host until the frame is done.
// Per queue entry: ray (64 B), path state (16 B); per path: one (emit, absorb) pair per scattering vertex (48 B)
// in a [bounce][path] stack, read back once when the path ends.
// ---------------------------------------------------------------------------------------------

constexpr uint32_t kMaxBounce = 128;  // deepest max_bounce a render call takes

struct WaveQueues {
    static constexpr size_t kLevel = 3;  // double2 per path and level of `stack`
    rtp_ray* rays[2];
    uint4* state[2];             // PathState::pack()
    WaveHit* hits;
    double2* stack;              // [bounce][path][3] double2: (emit.x, emit.y) (emit.z, absorb.x) (absorb.y, absorb.z)
    unsigned long long* count;   // [max_bounce + 1]
    size_t capacity;             // paths per launch the buffers were sized for (stride of `stack`)
    // path p's entry at level b of `stack`
    __device__ __forceinline__ double2* level(size_t b, size_t p) const { return stack + (b * capacity + p) * kLevel; }
};

// A path between two vertices, as its 16-byte queue record holds it: x = path index, y = next RNG draw,
// z = depth left | stack height << 8 | first-hit flag << 16
struct PathState {
    size_t p;  // 64-bit: held as 32 bits, it costs tail mode 48 B more of spill stores (ptxas, CUDA 12.9)
    uint32_t k, depth, nb, first_hit;
    __device__ __forceinline__ static PathState unpack(uint4 s) { return {s.x, s.y, s.z & 0xFFu, (s.z >> 8) & 0xFFu, (s.z >> 16) & 1u}; }
    __device__ __forceinline__ uint4 pack() const { return make_uint4(static_cast<uint32_t>(p), k, depth | (nb << 8) | (first_hit << 16), 0u); }
};

template <class Map>
__global__ void __launch_bounds__(256) wave_generate_kernel(DCamera cam, DRender rp, WaveQueues wq, size_t total, Map map) {
    const size_t p = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (p == 0) wq.count[0] = total;
    if (p >= total) return;
    uint32_t i, j;
    Rng rng = path_rng(rp, map, p, i, j);
    D3 o, d;
    primary_ray(cam, rp, i, j, rng, o, d);
    store_ray(wq.rays[0] + p, o, d);
    wq.state[0][p] = PathState{p, rng.k, rp.max_bounce, 0u, 0u}.pack();
}

// One vertex of a wavefront path (render.rs:102-131): the path's segment (o, d) missed (`miss`) or ended at h. `first`: the
// path's first segment, whose hit sets the foreground flag and, with fv != nullptr, records the vertex in *fv. A miss or a vertex
// that does not scatter ends the path with radiance L. A scattering vertex pushes (emit, absorb) onto the stack, leaves the
// scattered ray in (o, d) and spends one level of depth; at depth 0 the continuation returns black without tracing
// (render.rs:128-131), so L, black on entry, stays black. Returns whether the path lives on.
template <class Map>
__device__ __forceinline__ bool path_vertex(const DSceneView& sc, const DRender& rp, const Map& map, const WaveQueues& wq, PathState& s, bool first,
                                            bool miss, const HitRec& h, D3& o, D3& d, D3& L, FirstVertex* fv) {
    if (miss) {
        L = shade_miss(sc, d);
        return false;
    }
    if (first) s.first_hit = 1u;
    uint32_t i, j;
    Rng rng = path_rng(rp, map, s.p, i, j);
    rng.k = s.k;
    D3 emit, absorb;
    if (!shade_vertex(sc, o, d, h, rng, emit, absorb, first ? fv : nullptr)) {  // render.rs:108-110: emit + rgb(0,0,0)
        L = emit + mk(0.0, 0.0, 0.0);
        return false;
    }
    double2* sp = wq.level(s.nb, s.p);
    sp[0] = make_double2(emit.x, emit.y);
    sp[1] = make_double2(emit.z, absorb.x);
    sp[2] = make_double2(absorb.y, absorb.z);
    ++s.nb;
    s.depth -= 1;
    s.k = rng.k;
    return s.depth != 0;
}

// The end of a wavefront path whose last vertex left radiance L: render.rs:108-115 / 135-142, emit + absorb ⊙ (inner) folded
// inside-out like the recursion, into scratch[p] with the foreground flag
__device__ __forceinline__ void path_end(const WaveQueues& wq, const PathState& s, D3 L, double4* scratch) {
    for (int b = static_cast<int>(s.nb) - 1; b >= 0; --b) {
        const double2* sp = wq.level(b, s.p);
        const double2 s0 = sp[0], s1 = sp[1], s2 = sp[2];
        L = mk(s0.x, s0.y, s1.x) + cmul(mk(s1.y, s2.x, s2.y), L);
    }
    scratch[s.p] = make_double4(L.x, L.y, L.z, s.first_hit ? 1.0 : 0.0);
}

// A ray trace_any_kernel did not answer inside the wavefront integrator (not eligible for the f32 walk, stack overflow, abnormal leaf in
// the final window: a handful per frame at most) is marked in its hit record and traced here, by the thread that shades it, with the
// exact f64 walk of bvh.rs:93-119 (closest_hit_bvh): no second traversal launch per bounce.
constexpr uint32_t kDeferredHit = 0xFFFFFFFEu;
__device__ __noinline__ void trace_deferred(const DSceneView& sc, D3 o, D3 d, HitRec& h) {
    LocalCounters lc = {0, 0, 0, 0, 0, 0, 0};
    h.t = CUDART_INF; h.u = 0.0; h.v = 0.0; h.kind = 0;
    closest_hit_bvh<false>(sc, o, d, kRayEpsilon, h, lc);
}

constexpr int kShadeBlocks = 3;  // resident blocks per SM wave_shade_kernel is built for, and its grid
// With Aov::kOn the bounce-0 launch records every path's FirstVertex (its queue holds every path of the launch, hit or miss).
template <class Map, class Aov>
__global__ void __launch_bounds__(256, kShadeBlocks) wave_shade_kernel(DSceneView sc, DRender rp, WaveQueues wq, uint32_t bounce, double4* __restrict__ scratch,
                                                                       Map map, Aov aov) {
    const size_t n = static_cast<size_t>(wq.count[bounce]);
    const int cur = bounce & 1, nxt = cur ^ 1;
    const bool first = bounce == 0;
    const unsigned lane = threadIdx.x & 31u;
    const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
    // warp-uniform trip count: every lane of a warp takes part in the compaction ballot
    for (size_t q0 = (static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x) - lane; q0 < n; q0 += stride) {
        const size_t q = q0 + lane;
        bool alive = false;
        D3 o = mk(0, 0, 0), d = mk(0, 0, 0);
        uint4 st = make_uint4(0, 0, 0, 0);
        if (q < n) {
            const double2* rp2 = reinterpret_cast<const double2*>(wq.rays[cur] + q);
            const double2 r0 = rp2[0], r1 = rp2[1], r2 = rp2[2];
            o = mk(r0.x, r0.y, r1.x); d = mk(r1.y, r2.x, r2.y);
            PathState s = PathState::unpack(wq.state[cur][q]);
            const double2* hp = reinterpret_cast<const double2*>(wq.hits + q);
            const double2 h0 = hp[0], h1 = hp[1];
            uint32_t slotkind = static_cast<uint32_t>(__double2loint(h1.y));
            D3 L = mk(0.0, 0.0, 0.0);
            FirstVertex fv = {mk(0.0, 0.0, 0.0), mk(0.0, 0.0, 0.0)};
            HitRec h;
            h.t = h0.x; h.u = h0.y; h.v = h1.x; h.slot = slotkind & 0x7FFFFFFFu; h.kind = slotkind >> 31;
            if (slotkind == kDeferredHit) {
                trace_deferred(sc, o, d, h);
                slotkind = h.slot == kNoPrim ? kNoPrim : 0u;
            }
            alive = path_vertex(sc, rp, map, wq, s, first, slotkind == kNoPrim, h, o, d, L, Aov::kOn ? &fv : nullptr);
            if (!alive) path_end(wq, s, L, scratch);
            if (Aov::kOn && first) aov.record(s.p, fv);
            st = s.pack();
        }
        // compaction: survivors of this warp take consecutive slots of the next queue
        const unsigned live = __ballot_sync(0xffffffffu, alive);
        if (live) {
            const int leader = __ffs(live) - 1;
            unsigned long long base = 0;
            if (static_cast<int>(lane) == leader) base = atomicAdd(&wq.count[bounce + 1], static_cast<unsigned long long>(__popc(live)));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (alive) {
                const size_t dst = static_cast<size_t>(base) + __popc(live & ((1u << lane) - 1u));
                store_ray(wq.rays[nxt] + dst, o, d);
                wq.state[nxt][dst] = st;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// The persistent traversal kernel (state and steps: Walker above). Defined here because its tail mode shades in place.
// ---------------------------------------------------------------------------------------------

// Tail mode (OUT_TAIL) of the wavefront integrator: when a launch holds at most RTP_TAIL_THRESHOLD paths, one launch
// after generate carries every path of queue 0 to its end. A lane whose ray is finished shades it in place (path_vertex)
// and, if the path scattered, restarts its walker on the scattered ray, so the bounces cost one kernel instead of two
// launches each, and the culling tree stays warm in L1 across them. Results are the same bits: per path the
// sequence ray -> closest hit -> path_vertex is the one the trace/shade kernels perform.
struct TailArgs {
    WaveQueues q;
    DRender rp;
    double4* scratch;
};

constexpr int kTraceBlocksPerSM = 6;

// The in-order kernel: every lane walks in the reference's order (f32-eligible lanes on the 4-wide tree, the others on the exact f64
// pre-order tree). It serves List roots, scenes outside the any-order walk's preconditions, tail-mode launches, and the rays
// trace_any_kernel defers (index mode).
template <bool COUNT, int OUT, bool LIST>
__global__ void __launch_bounds__(128, OUT == OUT_TAIL ? 4 : kTraceBlocksPerSM) trace_persistent_kernel(DSceneView sc, const rtp_ray* __restrict__ rays, size_t n, void* __restrict__ out,
                                                                  Counters* counters, WorkQueue* wq, const unsigned long long* __restrict__ n_dev,
                                                                  TailArgs ta, DeferList index) {
    extern __shared__ __align__(16) uint32_t wide_stack[];  // [level][thread]
    if (n_dev) n = static_cast<size_t>(*n_dev);  // wavefront integrator: the batch size lives on the device
    if (index.idx) {
        // index mode: trace rays[index.idx[q]] for q < *index.count (deferred by trace_any_kernel). This launch is a programmatic
        // dependent of that kernel (launch_trace): its blocks may become resident while the last warps of trace_any_kernel still
        // walk, and wait here until that grid has completed and its writes are visible.
        asm volatile("griddepcontrol.wait;" ::: "memory");
        n = static_cast<size_t>(*index.count);
        // nothing deferred (the usual case): leave before touching the queue. trace_any_kernel's last warp has rearmed it and the
        // list is empty already, so there is nothing to reset; every warp reads the same final count, so every warp leaves. Two
        // same-address atomics per warp of this grid (queue claim, drain count) would otherwise delay the next launch.
        if (n == 0) return;
    }
    uint4 pst = make_uint4(0, 0, 0, 0);  // tail mode: the path state of the lane's ray (WaveQueues::state)
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    uint32_t* const my_stack = wide_stack + threadIdx.x;
    const uint32_t stride = blockDim.x;
    constexpr size_t kNoRay = ~static_cast<size_t>(0);
    LocalCounters lc = {0, 0, 0, 0, 0, 0, 0};

    // lane state: next == kEnd && prim == kNoPrim  -> empty (its finished ray, if any, is written at the next refill);
    //             prim != kNoPrim                  -> parked at a leaf;  otherwise walking
    Walker w;
    w.o = w.d = w.inv = mk(0, 0, 0);
    w.tmin = 0.0; w.h.t = 0.0; w.h.u = w.h.v = 0.0; w.h.slot = kNoPrim; w.h.kind = 0;
    w.next = kEnd; w.prim = kNoPrim; w.prim2 = kNoPrim; w.cur = 0; w.pend = 0; w.sp = 0; w.c0 = w.c1 = w.c2 = w.c3 = 0; w.onx = w.ony = w.onz = 0;
    w.fast = true; w.m32 = true; w.need_gate = false; w.sx = w.sy = w.sz = false;
    w.r32 = Ray32{0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    size_t idx = kNoRay;
    bool more = true;  // warp-uniform: the queue may still hold rays
    const size_t n_warps = static_cast<size_t>(gridDim.x) * (blockDim.x >> 5);
    const int lane_cap = static_cast<int>(min(static_cast<size_t>(32), max(static_cast<size_t>(kMinLanes), (n + n_warps - 1) / n_warps)));
    // refill at kRefillMin free lanes, or at half the cap of a warp that holds fewer rays. Written as a select: min(kRefillMin, ...)
    // is the same value, but with the constant folded in, ptxas (CUDA 12.9) gives <false, OUT_HIT, false> 36 B more of spill stores.
    const int refill_thr = lane_cap >= 2 * kRefillMin ? kRefillMin : max(1, lane_cap / 2);

    for (;;) {
        // ---- retire finished rays and refill ----------------------------------------------------------
        const bool is_done = (w.next == kEnd) & (w.prim == kNoPrim);
        const bool fin = OUT == OUT_TAIL && is_done && idx != kNoRay;  // tail mode: walk over, vertex not shaded yet
        const bool is_empty = is_done & !fin;
        const unsigned empty = __ballot_sync(0xffffffffu, is_empty);
        const int room = min(__popc(empty), max(lane_cap - (32 - __popc(empty)), 0));  // rays this warp may take now
        if (OUT == OUT_TAIL) {
            // shade finished rays in place; a path that scattered keeps its lane and walks on
            const unsigned finished = __ballot_sync(0xffffffffu, fin);
            if (finished != 0u && (__popc(finished) >= kPrimBatch || __ballot_sync(0xffffffffu, !is_done) == 0u)) {
                if (fin) {
                    PathState s = PathState::unpack(pst);
                    D3 L = mk(0.0, 0.0, 0.0), o = w.o, d = w.d;
                    // a path at full depth is on its first segment; tail mode serves rtp_render only: dense slots, no first vertex
                    const bool alive = path_vertex(sc, ta.rp, DenseTile{}, ta.q, s, s.depth == ta.rp.max_bounce, w.h.slot == kNoPrim, w.h, o, d, L, nullptr);
                    pst = s.pack();
                    if (alive) {
                        walker_start(w, sc, o, d, kRayEpsilon, CUDART_INF);
                        if (LIST) { w.m32 = false; if (sc.n_prims == 0) w.next = kEnd; }
                        lc.rays++;
                    } else {
                        path_end(ta.q, s, L, ta.scratch);
                        idx = kNoRay;
                    }
                }
                continue;
            }
        }
        if (empty == 0xffffffffu || (more && room >= refill_thr)) {
            if (OUT != OUT_TAIL && is_empty && idx != kNoRay) {
                write_hit<OUT>(sc, out, idx, w.o, w.d, w.h);
                idx = kNoRay;
            }
            if (!more) break;  // every lane is empty and the queue is drained
            // small batches are spread over all resident warps (fewer rays per warp, shorter critical path) instead of
            // filling a few warps to 32 lanes: a warp never holds more than lane_cap rays
            const int cnt = room, leader = __ffs(empty) - 1;
            unsigned long long base = 0;
            if (static_cast<int>(lane) == leader) base = atomicAdd(&wq->next, static_cast<unsigned long long>(cnt));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (base + static_cast<unsigned long long>(cnt) >= n) more = false;
            if (is_empty) {
                const int rank = __popc(empty & lt_mask);
                const size_t q = static_cast<size_t>(base) + rank;
                if (rank < cnt && q < n) {
                    const size_t i = index.idx ? static_cast<size_t>(index.idx[q]) : q;
                    idx = i;
                    const double2* rp = reinterpret_cast<const double2*>(rays + i);
                    const double2 r0 = __ldg(rp), r1 = __ldg(rp + 1), r2 = __ldg(rp + 2), r3 = __ldg(rp + 3);
                    walker_start(w, sc, mk(r0.x, r0.y, r1.x), mk(r1.y, r2.x, r2.y), r3.x, r3.y);
                    if (LIST) { w.m32 = false; if (sc.n_prims == 0) w.next = kEnd; }
                    if (OUT == OUT_TAIL) pst = ta.q.state[0][i];
                    lc.rays++;
                }
            }
            if (__ballot_sync(0xffffffffu, w.next != kEnd) == 0u) continue;
        }

        if (LIST) {
            // hittable.rs:110-120: every primitive, in caller order, no boxes
            if (w.next != kEnd) {
                const uint2 kp = __ldg(reinterpret_cast<const uint2*>(&sc.nodes[w.next].kind));  // kind, gate flag
                bool open = true;
                if (kp.y) {  // a leaf of a nested Bvh (bvh.rs:96): its own box first, with the current t_max
                    const double* pb = sc.prims[w.next].bmin;
                    const double2 b0 = ldg2(pb), b1 = ldg2(pb + 2), b2 = ldg2(pb + 4);
                    if (COUNT) lc.leaf_gates++;
                    open = w.fast ? collide_fast(b0, b1, b2, w.o, w.inv, w.sx, w.sy, w.sz, w.tmin, w.h.t) : collide_literal(b0, b1, b2, w.o, w.inv, w.tmin, w.h.t);
                }
                if (open) { w.prim = w.next | (kp.x << 31); w.need_gate = false; }
                w.next = w.next + 1 < sc.n_prims ? w.next + 1 : kEnd;
            }
        } else {
            // ---- hot walk: f32-eligible lanes take up to two steps per vote -----------------------------------
            for (;;) {
#pragma unroll
                for (int rep = 0; rep < 2; ++rep)  // measured: 3 or 4 steps per vote are slower in both walks
                    if ((w.next != kEnd) & (w.prim2 == kNoPrim) & w.m32) walker_step_wide<COUNT>(w, sc, lc, my_stack, stride);
                const unsigned walking = __ballot_sync(0xffffffffu, (w.next != kEnd) & (w.prim2 == kNoPrim) & w.m32);
                if (walking == 0u) break;
                const unsigned parked = __ballot_sync(0xffffffffu, w.prim != kNoPrim);
                if (__popc(parked) >= kPrimBatch) break;
                if (more && min(__popc(~(walking | parked)), max(lane_cap - __popc(walking | parked), 0)) >= refill_thr) break;
            }
            // ---- lanes outside the f32 path's preconditions take one exact step per round ------------------
            if (__any_sync(0xffffffffu, !w.m32)) {
                if ((w.next != kEnd) & (w.prim == kNoPrim) & !w.m32) walker_step64<COUNT>(w, sc, lc);
            }
        }

        // ---- leaves: exact gate + primitive test for the parked lanes --------------------------------
        if (w.prim != kNoPrim) {
            walker_leaf<COUNT>(w, sc, lc);
            // occlusion: T stays ray.t_max until the first accept, so that accept answers the ray (DESIGN.md §2c). The walk or
            // List scan ends and the second pending leaf is dropped; the lane retires at the next refill.
            if (OUT == OUT_OCCLUDED && w.h.slot != kNoPrim) { w.next = kEnd; w.prim = kNoPrim; }
        }
    }

    flush_counters<COUNT>(counters, lc);
    // the last warp to drain rearms the queue, so back-to-back launches need no memset (no block barrier: warps leave
    // as soon as they are done)
    if (lane == 0) {
        __threadfence();
        if (atomicAdd(&wq->done_blocks, 1u) == static_cast<unsigned>(n_warps) - 1u) {
            wq->next = 0ull;
            wq->done_blocks = 0u;
            if (index.idx) *index.count = 0ull;  // the deferred rays are done: rearm the list for the next launch
            __threadfence();
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Pure any-order traversal kernel (DESIGN.md 4b/6). The walk of DESIGN.md 4b (nearest child first, distance culling against a
// window), built around what the profile of round 1's combined in-order/any-order kernel showed (profiles/r01_trace_any_c2.md: 14 % of the executed
// instructions were register moves at loop heads, 19 % branch / reconvergence / predicate set-up, 12 % the slab arithmetic):
//   * one loop with one back edge; lane state is a handful of scalars (node, stack top as a shared-memory ADDRESS, two pending
//     leaf words), no struct passed by reference through inlined functions with early returns;
//   * only any-order lanes live here. A ray that is not eligible (axis-parallel, non-finite, huge coordinates, t_min < 0), whose
//     stack would overflow, or whose answer may depend on the reference's visiting order (abnormal leaf inside the final
//     window) is appended to a DEFER list and traced by a second launch of the in-order kernel (trace_persistent_kernel with an
//     index list), so neither the in-order walker nor the exact f64 walker is compiled into this kernel;
//   * the scene's big primitives (at most eight) are tested when the ray starts, with all lanes of the refill together, instead
//     of travelling through the tree as window-exempt children: the step carries no big-mask load and no per-child selects,
//     and the walk starts with the window already closed to the nearest big hit. Testing them first is the same sequential
//     process (the claim in DESIGN.md 4b does not depend on the order in which leaves are looked at); a big leaf met again in
//     the rank-ordered tree is skipped (kWideBig), the order-free tree has none. A ray whose window then closes before the
//     culled-set box (every other leaf) is finished without a walk;
//   * rays are read with ld.global.nc.L1::no_allocate and results written with st.global.cs: the 80 B/ray stream does not
//     displace the culling tree from L1.
// ---------------------------------------------------------------------------------------------

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void sts_v2(uint32_t addr, uint32_t a, uint32_t b) { asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(addr), "r"(a), "r"(b) : "memory"); }
__device__ __forceinline__ uint2 lds_v2(uint32_t addr) {
    uint2 r;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(r.x), "=r"(r.y) : "r"(addr) : "memory");
    return r;
}
__device__ __forceinline__ uint4 lds_v4(uint32_t addr) {
    uint4 r;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr) : "memory");
    return r;
}
__device__ __forceinline__ void sts_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t r;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r) : "r"(addr) : "memory");
    return r;
}
__device__ __forceinline__ void sts_u32(uint32_t addr, uint32_t a) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(a) : "memory"); }
__device__ __forceinline__ uint32_t dlo(double x) { return static_cast<uint32_t>(__double2loint(x)); }
__device__ __forceinline__ uint32_t dhi(double x) { return static_cast<uint32_t>(__double2hiint(x)); }
__device__ __forceinline__ double mkd(uint32_t lo, uint32_t hi) { return __hiloint2double(static_cast<int>(hi), static_cast<int>(lo)); }
__device__ __forceinline__ double2 ldg_stream2(const double* p) {
    double2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p));
    return r;
}

constexpr uint32_t kAnyStride = 128u * 8u;  // bytes between two levels of a thread's stack column ([entry][thread] of uint2)
// The part of a lane's state that only a hit, the set-up and the retirement touch lives in shared memory behind the stacks, as four
// [chunk][thread] words of 16 bytes (conflict-free ld/st.shared.v4): 14 registers less in the walk, which is what lets six blocks
// share an SM without spills.  0: 1/d.x, 1/d.y   1: 1/d.z, slack s0, slack s1 (floats)   2: best u, best v
// 3: smallest abnormal t (float bits), ray index (0xFFFFFFFF: the lane holds no ray), -, -
constexpr uint32_t kColdStride = 128u * 16u;
constexpr size_t kAnyColdBytes = static_cast<size_t>(kColdStride) * 4u;

// per-ray eligibility and slack coefficients (DESIGN.md §4, 4b) from scalars; false: the ray goes to the in-order kernel.
// Everything is evaluated in f32 with every operation rounded up (all quantities are non-negative), so the slack is an upper bound of
// the real-number expression in DESIGN.md 4b; the magnitudes are converted first and maximised in f32 (RU is monotone, so that
// equals converting the f64 maximum), which also serves the range checks of the f32 walk: finite origin with |o| <= 1e15 and
// 1e-15 <= |1/d| <= 1e15 on every axis (the float thresholds sit just inside the f64 ones, and a NaN fails every comparison).
__device__ __forceinline__ bool any_slack_of(const DSceneView& sc, D3 o, D3 d, D3 inv, double tmin, float& s0f, float& s1f) {
    const float u = 0x1.0p-53f, K = 8.9e-9f;  // K >= 8 u 1e7: |det| >= 1e-7 (hittable.rs:80), 8u: rounding of a 6-term sum of products
    const float Po = fmaxf(fmaxf(__double2float_ru(fabs(o.x)), __double2float_ru(fabs(o.y))), __double2float_ru(fabs(o.z)));
    const float D = fmaxf(fmaxf(__double2float_ru(fabs(d.x)), __double2float_ru(fabs(d.y))), __double2float_ru(fabs(d.z)));
    const float I = fmaxf(fmaxf(__double2float_ru(fabs(inv.x)), __double2float_ru(fabs(inv.y))), __double2float_ru(fabs(inv.z)));
    const float Imin = fminf(fminf(__double2float_rd(fabs(inv.x)), __double2float_rd(fabs(inv.y))), __double2float_rd(fabs(inv.z)));
    const bool in_range = (Po <= 1e15f) & (I <= 1e15f) & (Imin >= 1.0000001e-15f);
    const float P = __fadd_ru(Po, sc.any_Af);
    const float E = sc.any_Ef;
    const float E2 = __fmul_ru(E, E), DE2 = __fmul_ru(D, E2), PE = __fmul_ru(P, E);
    const float kappa = __fmul_ru(__fmul_ru(K, 6.0f), DE2);
    const float e_uv = __fadd_ru(__fmul_ru(K, __fadd_ru(__fmul_ru(6.0f, __fmul_ru(PE, D)), __fmul_ru(6.06f, DE2))), 3.0f * u);
    const float eta = __fmul_ru(__fadd_ru(__fmul_ru(4.0f, e_uv), 5.0f * u), E);
    // 1 / (1 - kappa) <= 4/3 for kappa <= 1/4: no divide on the per-ray path; the factor 4 in front absorbs the second-order terms
    const float a0 = __fmul_ru(__fmul_ru(__fadd_ru(eta, __fmul_ru(u, P)), I), 1.0000002f);
    const float a1 = __fmul_ru(__fmul_ru(__fmul_ru(K, 6.0f), __fmul_ru(PE, E)), 1.3333334f);
    const float a2 = __fmul_ru(3.0f * u, __double2float_ru(fabs(tmin)));
    float a3 = 0.f;
    if (sc.any_Rf >= 0.f) {  // scene-uniform branch: spheres that are not big (DESIGN.md 4b "Spheres")
        const float oc = __fadd_ru(Po, sc.any_Cf);
        const float S = __fadd_ru(__fmul_ru(3.0f, __fmul_ru(oc, oc)), __fmul_ru(sc.any_Rf, sc.any_Rf));
        const float g = __fsqrt_ru(__fmul_ru(40.0f * u, S));
        a3 = __fmul_ru(__fadd_ru(__fmul_ru(3.0f, g), __fmul_ru(u, __fadd_ru(__fmul_ru(2.0f, __fadd_ru(sc.any_Cf, sc.any_Rf)), oc))), I);
    }
    s0f = __fmul_ru(4.0f, __fadd_ru(__fadd_ru(__fadd_ru(a0, a1), a2), a3));
    s1f = __fmul_ru(4.0f, __fadd_ru(__fmul_ru(__fadd_ru(__fmul_ru(__fmul_ru(K, 6.0f), DE2), 5.0f * u), 1.3333334f), 8.0f * u));
    return in_range & (kappa <= 0.25f) & (e_uv <= 0.01f) & (s0f <= 3.0e38f) & (s1f <= 3.0e38f);
}

constexpr int kAnyBlocks = 6;    // resident blocks per SM the kernel is built for (register budget 65536 / (128 x blocks))
constexpr int kAnySteps = 2;     // walk steps per round of votes
constexpr int kAnyPrefetch = 2;  // L2 prefetch distance of the ray stream, in quarters of (warps of the grid) x (rays per reservation)
constexpr int kAnyPopLoop = 2;   // stack entries a step may take before it visits a node (1: one per step, as in the first version)

template <bool COUNT, int OUT>
__global__ void __launch_bounds__(128, kAnyBlocks) trace_any_kernel(DSceneView sc, const rtp_ray* __restrict__ rays, size_t n, void* __restrict__ out, Counters* counters,
                                                       WorkQueue* wq, const unsigned long long* __restrict__ n_dev, DeferList defer) {
    extern __shared__ __align__(16) uint32_t any_stack[];
    // the launch over the defer list (launch_trace) may be set up while this grid runs: it waits for this grid's completion itself
    asm volatile("griddepcontrol.launch_dependents;");
    if (n_dev) n = static_cast<size_t>(*n_dev);
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    const uint32_t sbase = smem_u32(any_stack) + threadIdx.x * 8u;      // bottom of this thread's stack column
    const uint32_t slimit = sbase + (sc.any_cap - 3u) * kAnyStride;     // pushing three more entries above this would overflow
    const uint32_t cold = smem_u32(any_stack) + sc.any_cap * kAnyStride + threadIdx.x * 16u;  // chunk 0 of this thread's cold state
    LocalCounters lc = {0, 0, 0, 0, 0, 0, 0};
    sts_v4(cold + 3u * kColdStride, __float_as_uint(CUDART_INF_F), 0xFFFFFFFFu, 0u, 0u);

    // ---- lane state in registers (1/d, the slack coefficients, best u and v, the abnormal mark and the ray index are cold) ---------
    D3 o = mk(0, 0, 0), d = mk(0, 0, 0);
    double tmin = 0.0;
    double best_t = 0.0;                              // t of the closest normal hit so far (valid when best != kNoPrim)
    uint32_t best = kNoPrim;                          // slot | kind << 31
    double T_win = 0.0;                               // window top: min(ray.t_max, best_t + 2 slack(best_t))
    float ix = 0.f, iy = 0.f, iz = 0.f, clx = 0.f, cly = 0.f, clz = 0.f, chx = 0.f, chy = 0.f, chz = 0.f, tmin_dn = 0.f, T_up = 0.f;
    uint32_t onx = 0, ony = 2, onz = 4;  // float4 index of the near plane of each axis inside a node (DWide::plane); the far plane is that index ^ 1
    bool sx = false, sy = false, sz = false;
    uint32_t node = kNone;        // node to visit next, or kNone: take the next stack entry
    uint32_t sp = sbase;          // shared-memory address of the first free entry of this thread's column
    uint32_t leaf0 = 0u, leaf1 = 0u;  // pending leaves (raw child words, oldest first); 0 = none (child word 0 is the root, never a leaf)
    bool more = true;             // warp-uniform: the queue may still hold rays
    const size_t n_warps = static_cast<size_t>(gridDim.x) * (blockDim.x >> 5);
    const int lane_cap = static_cast<int>(min(static_cast<size_t>(32), max(static_cast<size_t>(kMinLanes), (n + n_warps - 1) / n_warps)));
    const int refill_thr = lane_cap >= 2 * kRefillMin ? kRefillMin : max(1, lane_cap / 2);
    const float4* __restrict__ tree = reinterpret_cast<const float4*>(sc.any_wide);  // a node = 8 float4: 32-bit indexing (device_scene_upload: < 2^29 nodes)

    // exact test of one leaf in any-order mode
    auto test_leaf = [&](uint32_t cw) {
        const uint32_t slot = cw & kWideSlotMask, kind = (cw >> 30) & 1u;
        const DPrim* p = sc.prims + slot;
        double t, u = 0.0, v = 0.0;
        bool hit;
        if (kind == RTP_HITTABLE_TRIANGLE) {
            if (COUNT) lc.triangle_tests++;
            hit = test_triangle(p, o, d, tmin, T_win, t, u, v);
        } else {
            if (COUNT) lc.sphere_tests++;
            hit = test_sphere(p, o, d, tmin, T_win, t);
        }
        if (hit) {
            if (!(t == t)) {
                sts_u32(cold + 3u * kColdStride, __float_as_uint(-CUDART_INF_F));  // NaN t (overflowing geometry): let the in-order walk decide
            } else {
                const uint4 c0 = lds_v4(cold), c1 = lds_v4(cold + kColdStride);
                const D3 inv = mk(mkd(c0.x, c0.y), mkd(c0.z, c0.w), mkd(c1.x, c1.y));
                const double* pb = p->bmin;
                const double2 b0 = ldg2(pb), b1 = ldg2(pb + 2), b2 = ldg2(pb + 4);
                if (COUNT) lc.leaf_gates++;
                if (collide_fast(b0, b1, b2, o, inv, sx, sy, sz, tmin, t)) {
                    // normal leaf: min t, ties to the larger DFS rank (= slot)
                    const uint32_t bslot = best & 0x7FFFFFFFu;
                    if (best == kNoPrim || t < best_t || (t == best_t && slot > bslot)) {
                        best_t = t; best = slot | (kind << 31);
                        sts_v4(cold + 2u * kColdStride, dlo(u), dhi(u), dlo(v), dhi(v));
                        const double win = t + 2.0 * (static_cast<double>(__uint_as_float(c1.z)) + static_cast<double>(__uint_as_float(c1.w)) * fabs(t));
                        T_win = fmin(T_win, win);
                        T_up = __double2float_ru(T_win);
                    }
                } else if (collide_fast(b0, b1, b2, o, inv, sx, sy, sz, tmin, CUDART_INF)) {
                    // abnormal: its box is entered, but only after t (rounded DOWN to f32: conservative)
                    const float a_min = __uint_as_float(lds_u32(cold + 3u * kColdStride));
                    sts_u32(cold + 3u * kColdStride, __float_as_uint(fminf(a_min, __double2float_rd(t))));
                }
            }
        }
    };

    for (;;) {
        // ---- retire finished rays and refill ------------------------------------------------------------------------------
        const bool walking0 = (node != kNone) | (sp != sbase);
        const bool busy = walking0 | (leaf0 != 0u);
        const unsigned busy_mask = __ballot_sync(0xffffffffu, busy);
        const int n_busy = __popc(busy_mask);
        const int room = min(32 - n_busy, max(lane_cap - n_busy, 0));
        if (busy_mask == 0u || (more && room >= refill_thr)) {
            const uint4 c3 = lds_v4(cold + 3u * kColdStride);
            const uint32_t idx = c3.y;              // ray held by this lane (index into rays / out), 0xFFFFFFFF = none
            if (!busy && idx != 0xFFFFFFFFu) {
                const float A_min = __uint_as_float(c3.x);
                // the walk of this lane's ray is over. An abnormal leaf inside the final window: the answer may depend on the
                // reference's visiting order, the in-order kernel decides (A_min was rounded down, T_win compared in f64: conservative)
                if (A_min != CUDART_INF_F && static_cast<double>(A_min) <= T_win) {
                    if (OUT == OUT_WAVE) {  // the thread that shades this vertex traces it with the exact walk (wave_shade_kernel)
                        reinterpret_cast<double2*>(static_cast<WaveHit*>(out) + idx)[1] = make_double2(0.0, __hiloint2double(0, static_cast<int>(kDeferredHit)));
                    } else {
                        const unsigned long long slot = atomicAdd(defer.count, 1ull);
                        defer.idx[slot] = idx;
                        lc.rays--;  // the in-order kernel counts it
                    }
                    if (COUNT) lc.rewalks++;
                } else {
                    const uint4 c2 = lds_v4(cold + 2u * kColdStride);
                    HitRec h;
                    h.t = best_t; h.u = mkd(c2.x, c2.y); h.v = mkd(c2.z, c2.w); h.slot = best == kNoPrim ? kNoPrim : (best & 0x7FFFFFFFu); h.kind = best >> 31;
                    write_hit<OUT>(sc, out, idx, o, d, h);
                }
                sts_u32(cold + 3u * kColdStride + 4u, 0xFFFFFFFFu);
            }
            if (!more) {
                if (busy_mask == 0u) break;
            } else {
                const unsigned free_mask = ~busy_mask;
                const int cnt = room, leader = __ffs(free_mask) - 1;
                unsigned long long base = 0;
                if (static_cast<int>(lane) == leader) base = atomicAdd(&wq->next, static_cast<unsigned long long>(cnt));
                base = __shfl_sync(0xffffffffu, base, leader);
                if (base + static_cast<unsigned long long>(cnt) >= n) more = false;
                const int rank = __popc(free_mask & lt_mask);
                // the ray stream comes from HBM and the first thing a refill does with a ray is divide by its direction: pull the
                // rays some warp will take about one refill from now into L2 (a quarter of the grid's warps x 32 rays up the queue
                // per unit of kAnyPrefetch). Stateless: the queue is handed out in order, whoever takes them finds them there.
                const unsigned long long pf = base + static_cast<unsigned long long>(kAnyPrefetch) * (n_warps / 4) * 32ull + static_cast<unsigned>(rank);
                if (!busy && rank < cnt && pf < n) asm volatile("prefetch.global.L2 [%0];" ::"l"(rays + pf));
                const uint32_t i = (!busy && rank < cnt && base + static_cast<unsigned>(rank) < n) ? static_cast<uint32_t>(base) + static_cast<uint32_t>(rank) : 0xFFFFFFFFu;
                if (i != 0xFFFFFFFFu) {
                    const double* rp = reinterpret_cast<const double*>(rays + i);
                    const double2 r0 = ldg_stream2(rp), r1 = ldg_stream2(rp + 2), r2 = ldg_stream2(rp + 4), r3 = ldg_stream2(rp + 6);
                    o = mk(r0.x, r0.y, r1.x); d = mk(r1.y, r2.x, r2.y);
                    tmin = r3.x;
                    const double tmax = r3.y;
                    const D3 inv = mk(1.0 / d.x, 1.0 / d.y, 1.0 / d.z);  // utility.rs:71-77 Ray::expand
                    float s0f, s1f;
                    // eligibility: finite origin, 1e-15 <= |1/d| <= 1e15 on every axis, |o| <= 1e15 and a self-consistent slack
                    // (any_slack_of), 0 <= t_min <= t_max
                    const bool ok = any_slack_of(sc, o, d, inv, tmin, s0f, s1f) & (tmax >= tmin) & (tmin >= 0.0);
                    if (ok || OUT == OUT_WAVE) lc.rays++;  // a ray deferred to the in-order kernel is counted there
                    if (!ok) {
                        if (OUT == OUT_WAVE) {
                            reinterpret_cast<double2*>(static_cast<WaveHit*>(out) + i)[1] = make_double2(0.0, __hiloint2double(0, static_cast<int>(kDeferredHit)));
                        } else {
                            const unsigned long long slot = atomicAdd(defer.count, 1ull);
                            defer.idx[slot] = i;
                        }
                    } else {
                        sts_v4(cold, dlo(inv.x), dhi(inv.x), dlo(inv.y), dhi(inv.y));
                        sts_v4(cold + kColdStride, dlo(inv.z), dhi(inv.z), __float_as_uint(s0f), __float_as_uint(s1f));
                        sts_v4(cold + 2u * kColdStride, 0u, 0u, 0u, 0u);
                        sts_v4(cold + 3u * kColdStride, __float_as_uint(CUDART_INF_F), i, 0u, 0u);
                        sx = inv.x < 0.0; sy = inv.y < 0.0; sz = inv.z < 0.0;
                        const double px = o.x * inv.x, py = o.y * inv.y, pz = o.z * inv.z;
                        const double kx = fabs(px) * 0x1.0p-21 + 1e-37, ky = fabs(py) * 0x1.0p-21 + 1e-37, kz = fabs(pz) * 0x1.0p-21 + 1e-37;
                        ix = __double2float_rn(inv.x); iy = __double2float_rn(inv.y); iz = __double2float_rn(inv.z);
                        clx = __double2float_rd(-px - kx); cly = __double2float_rd(-py - ky); clz = __double2float_rd(-pz - kz);
                        chx = __double2float_ru(-px + kx); chy = __double2float_ru(-py + ky); chz = __double2float_ru(-pz + kz);
                        tmin_dn = __double2float_rd(tmin);
                        onx = sx ? 1u : 0u; ony = sy ? 3u : 2u; onz = sz ? 5u : 4u;
                        best = kNoPrim; best_t = tmax;
                        T_win = tmax; T_up = __double2float_ru(tmax);
                        leaf0 = 0u; leaf1 = 0u; sp = sbase;
                        // the big primitives first, all lanes of the refill together
                        for (uint32_t k = 0; k < sc.n_big; ++k) test_leaf(kWideLeaf | ((sc.big[k] >> 31) << 30) | (sc.big[k] & kWideSlotMask));
                        // then the culled-set box (every leaf that is not big lies inside it) against the window those tests left, with
                        // the node test's arithmetic: rejected, the ray is done without a walk (most primary rays of the bunny scenes
                        // end on the ground sphere in front of the bunny's box)
                        const float cn = fmaxf(fmaxf(fmaf(sx ? sc.cull[3] : sc.cull[0], ix, clx), fmaf(sy ? sc.cull[4] : sc.cull[1], iy, cly)),
                                               fmaxf(fmaf(sz ? sc.cull[5] : sc.cull[2], iz, clz), tmin_dn));
                        const float cf = fminf(fminf(fmaf(sx ? sc.cull[0] : sc.cull[3], ix, chx), fmaf(sy ? sc.cull[1] : sc.cull[4], iy, chy)),
                                               fminf(fmaf(sz ? sc.cull[2] : sc.cull[5], iz, chz), T_up));
                        node = cf >= cn ? 0u : kNone;
                    }
                }
            }
        }

        if (COUNT) {
            const bool cw = (leaf1 == 0u) & ((node != kNone) | (sp != sbase));
            const unsigned m_walk = __ballot_sync(0xffffffffu, cw), m_full = __ballot_sync(0xffffffffu, leaf1 != 0u);
            const unsigned m_wait = __ballot_sync(0xffffffffu, !cw & (leaf0 != 0u) & (leaf1 == 0u));
            const unsigned m_empty = __ballot_sync(0xffffffffu, !cw & (leaf0 == 0u));
            if (lane == 0 && counters) {
                atomicAdd(&counters->rounds, 1ull); atomicAdd(&counters->lanes_walk, static_cast<unsigned long long>(__popc(m_walk)));
                atomicAdd(&counters->lanes_full, static_cast<unsigned long long>(__popc(m_full))); atomicAdd(&counters->lanes_leafwait, static_cast<unsigned long long>(__popc(m_wait)));
                atomicAdd(&counters->lanes_empty, static_cast<unsigned long long>(__popc(m_empty)));
            }
        }
        // ---- which phase: when more lanes wait for a leaf test than can walk, test leaves first (incoherent rays: a few long walks
        //      would otherwise run at a handful of lanes while most of the warp waits for its primitive tests) ---------------------
        bool leaf_first = false;
        {
            const int n_walk = __popc(__ballot_sync(0xffffffffu, (leaf1 == 0u) & ((node != kNone) | (sp != sbase))));
            const int n_leaf = __popc(__ballot_sync(0xffffffffu, leaf0 != 0u));
            leaf_first = n_leaf >= kPrimBatch && n_leaf > n_walk;
        }
        // ---- walk: up to two steps per round ----------------------------------------------------------------------------------
        if (!leaf_first) {
#pragma unroll
        for (int rep = 0; rep < kAnySteps; ++rep) {
            if ((leaf1 == 0u) & ((node != kNone) | (sp != sbase))) {
                // take postponed entries until one gives a node to visit: leaves go to the pending pair, entries beyond the window are
                // dropped. (One entry per step left half of the step slots of incoherent rays without a node: RTP_LANE_STATS; an
                // unbounded loop runs its late iterations for three or four lanes: kAnyPopLoop bounds the pops per step.)
#pragma unroll 1
                for (int pops = 0; pops < kAnyPopLoop && ((node == kNone) & (sp != sbase) & (leaf1 == 0u)); ++pops) {
                    sp -= kAnyStride;
                    const uint2 e = lds_v2(sp);
                    const bool inside = __uint_as_float(e.y) <= T_up;  // else: the window shrank since this entry was postponed
                    const bool is_leaf = (e.x & kWideLeaf) != 0u;
                    const bool first = leaf0 == 0u;
                    node = (inside & !is_leaf) ? e.x : kNone;
                    leaf1 = (inside & is_leaf & !first) ? e.x : leaf1;
                    leaf0 = (inside & is_leaf & first) ? e.x : leaf0;
                }
                if (node != kNone) {
                    const uint32_t nb = node * 8u;
                    const float4 nx4 = __ldg(tree + (nb + onx));
                    const float4 ny4 = __ldg(tree + (nb + ony));
                    const float4 nz4 = __ldg(tree + (nb + onz));
                    const float4 fx4 = __ldg(tree + ((nb + onx) ^ 1u));
                    const float4 fy4 = __ldg(tree + ((nb + ony) ^ 1u));
                    const float4 fz4 = __ldg(tree + ((nb + onz) ^ 1u));
                    const uint4 ch = __ldg(reinterpret_cast<const uint4*>(tree + (nb + 6u)));
                    // key = conservative entry distance (non-negative float: its bits order like the value) with the child index in the
                    // two low bits; a child that is missed, beyond the window or empty gets the largest key
#define RTP_KEY(c, idx_)                                                                                                            \
    const float n##c = fmaxf(fmaxf(fmaf(nx4.c, ix, clx), fmaf(ny4.c, iy, cly)), fmaxf(fmaf(nz4.c, iz, clz), tmin_dn));               \
    const float f##c = fminf(fminf(fmaf(fx4.c, ix, chx), fmaf(fy4.c, iy, chy)), fminf(fmaf(fz4.c, iz, chz), T_up));                  \
    const uint32_t k##c = f##c >= n##c ? ((__float_as_uint(n##c) & ~3u) | idx_) : 0xFFFFFFFFu;
                    RTP_KEY(x, 0u) RTP_KEY(y, 1u) RTP_KEY(z, 2u) RTP_KEY(w, 3u)
#undef RTP_KEY
                    if (COUNT) {
                        lc.node_visits++;
                        const double* b64 = sc.any_boxes + static_cast<size_t>(node) * 24;
                        const uint32_t keys[4] = {kx, ky, kz, kw};
                        const uint4 c0 = lds_v4(cold), c1 = lds_v4(cold + kColdStride);
                        const D3 inv = mk(mkd(c0.x, c0.y), mkd(c0.z, c0.w), mkd(c1.x, c1.y));
                        for (uint32_t k = 0; k < 4; ++k)  // a rejected child must fail the exact test with the window top as t_max
                            if (keys[k] == 0xFFFFFFFFu && (&ch.x)[k] != kWideEmpty &&
                                collide_literal(ldg2(b64 + 6 * k), ldg2(b64 + 6 * k + 2), ldg2(b64 + 6 * k + 4), o, inv, tmin, T_win))
                                lc.violations++;
                    }
                    const uint32_t a0 = min(kx, ky), a1 = max(kx, ky), b0 = min(kz, kw), b1 = max(kz, kw);
                    uint32_t s0 = min(a0, b0);
                    const uint32_t m0 = max(a0, b0), m1 = min(a1, b1), s3 = max(a1, b1);
                    const uint32_t s1 = min(m0, m1), s2 = max(m0, m1);
#define RTP_SEL(k) (((k) & 2u) ? (((k) & 1u) ? ch.w : ch.z) : (((k) & 1u) ? ch.y : ch.x))
                    node = kNone;
                    {
                        // the three farther children, farthest first, without branches: every lane writes its three candidate entries
                        // at consecutive positions and advances the stack top only past the ones that exist (the keys are sorted:
                        // an absent child is never followed by a present one). Incoherent rays ran the nested pushes at 2-7 lanes.
                        const bool p1 = s1 != 0xFFFFFFFFu, p2 = s2 != 0xFFFFFFFFu, p3 = s3 != 0xFFFFFFFFu;
                        if (p1 & (sp > slimit)) {
                            // no room to postpone three children: give the ray to the in-order kernel
                            sts_u32(cold + 3u * kColdStride, __float_as_uint(-CUDART_INF_F)); sp = sbase; leaf0 = 0u; leaf1 = 0u; s0 = 0xFFFFFFFFu;
                        } else {
                            const uint32_t a3 = sp, a2 = a3 + (p3 ? kAnyStride : 0u), a1 = a2 + (p2 ? kAnyStride : 0u);
                            if (p3) sts_v2(a3, RTP_SEL(s3), s3 & ~3u);
                            if (p2) sts_v2(a2, RTP_SEL(s2), s2 & ~3u);
                            if (p1) sts_v2(a1, RTP_SEL(s1), s1 & ~3u);
                            sp = a1 + (p1 ? kAnyStride : 0u);
                        }
                    }
                    {   // the nearest child: a node is visited next, a leaf joins the pending pair; selects only
                        const uint32_t c = RTP_SEL(s0);
                        const bool valid = s0 != 0xFFFFFFFFu, is_leaf = (c & kWideLeaf) != 0u, first = leaf0 == 0u;
                        node = (valid & !is_leaf) ? c : kNone;
                        leaf1 = (valid & is_leaf & !first) ? c : leaf1;
                        leaf0 = (valid & is_leaf & first) ? c : leaf0;
                    }
#undef RTP_SEL
                }
            }
        }
        }

        // ---- leaves: when enough lanes hold one, or nobody can walk ----------------------------------------------------------
        const unsigned parked = __ballot_sync(0xffffffffu, leaf0 != 0u);
        if (parked != 0u) {
            const unsigned walking = __ballot_sync(0xffffffffu, (leaf1 == 0u) & ((node != kNone) | (sp != sbase)));
            if (__popc(parked) >= kPrimBatch || walking == 0u) {
                if (COUNT && lane == 0 && counters) { atomicAdd(&counters->leaf_rounds, 1ull); atomicAdd(&counters->leaf_lanes, static_cast<unsigned long long>(__popc(parked))); }
                if (leaf0 != 0u) {
                    if (!(leaf0 & kWideBig)) test_leaf(leaf0);  // big primitives were tested when the ray started
                    leaf0 = leaf1;
                    leaf1 = 0u;
                }
            }
        }
    }

    flush_counters<COUNT>(counters, lc);
    if (lane == 0) {
        __threadfence();
        if (atomicAdd(&wq->done_blocks, 1u) == static_cast<unsigned>(n_warps) - 1u) {
            wq->next = 0ull;
            wq->done_blocks = 0u;
            __threadfence();
        }
    }
}

// FP64 throughput probe (rtp_probe_fp64): eight independent multiply-then-add chains per thread; with --fmad=false each step
// is one DMUL and one DADD, the instruction mix of the path itself
__global__ void __launch_bounds__(256) fp64_probe_kernel(double* __restrict__ sink, double a, double b, int iters) {
    double x[8];
    for (int k = 0; k < 8; ++k) x[k] = 1.0 + 1e-3 * (threadIdx.x + k);
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 8; ++k) x[k] = x[k] * a + b;
    }
    double s = 0.0;
    for (int k = 0; k < 8; ++k) s += x[k];
    if (s == 123.456) sink[blockIdx.x] = s;  // never true: keeps the chains alive
}

// main.rs:78-87: per pixel, add the samples of this launch in sample order to the running sums; on the
// last launch optionally divide by num_samples. acc is (r,g,b,foreground) per tile pixel.
__global__ void __launch_bounds__(256) resolve_kernel(const double4* __restrict__ scratch, double4* __restrict__ acc, size_t npix, uint32_t n_samples,
                                                       int first_launch) {
    const size_t pix = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (pix >= npix) return;
    double4 a = first_launch ? make_double4(0.0, 0.0, 0.0, 0.0) : acc[pix];
    for (uint32_t s = 0; s < n_samples; ++s) {
        const double4 c = scratch[pix * n_samples + s];  // path_rng: the samples of a pixel are adjacent
        a.x += c.x; a.y += c.y; a.z += c.z; a.w += c.w;
    }
    acc[pix] = a;
}

// the frame pixel of tile pixel `pix` of a launch (row-major over the launch's rows, rp.tile_w wide): the output kernels' mapping
__device__ __forceinline__ size_t frame_pixel(const DRender& rp, size_t pix) {
    const uint32_t i = rp.tile_x + static_cast<uint32_t>(pix % rp.tile_w);
    const uint32_t j = rp.tile_y + rp.row_offset + static_cast<uint32_t>(pix / rp.tile_w) * rp.row_stride;
    return static_cast<size_t>(i) + static_cast<size_t>(j) * rp.width;
}

__global__ void __launch_bounds__(256) write_frame_kernel(const double4* __restrict__ acc, DRender rp, double divisor, double* __restrict__ rgb,
                                                           double* __restrict__ fg) {
    const size_t npix = static_cast<size_t>(rp.tile_w) * rp.tile_h;
    const size_t pix = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (pix >= npix) return;
    const size_t px = frame_pixel(rp, pix);
    double4 a = acc[pix];
    if (divisor != 0.0) { a.x = a.x / divisor; a.y = a.y / divisor; a.z = a.z / divisor; a.w = a.w / divisor; }
    rgb[3 * px + 0] = a.x; rgb[3 * px + 1] = a.y; rgb[3 * px + 2] = a.z;
    if (fg) fg[px] = a.w;
}

// rtp_render_aov (DESIGN.md §6c): resolve_kernel for the launch's AovRecords. acc is 3 double2 per tile pixel, (albedo, normal)
// summed from 0.0 in sample order like the colour.
__global__ void __launch_bounds__(256) aov_resolve_kernel(const double2* __restrict__ rec, double2* __restrict__ acc, size_t npix, uint32_t n_samples,
                                                           int first_launch) {
    const size_t pix = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (pix >= npix) return;
    double2 a0 = make_double2(0.0, 0.0), a1 = a0, a2 = a0;
    if (!first_launch) { a0 = acc[3 * pix]; a1 = acc[3 * pix + 1]; a2 = acc[3 * pix + 2]; }
    for (uint32_t s = 0; s < n_samples; ++s) {
        const double2* r = rec + 3 * (pix * n_samples + s);  // path_rng: the samples of a pixel are adjacent
        const double2 r0 = r[0], r1 = r[1], r2 = r[2];
        a0.x += r0.x; a0.y += r0.y; a1.x += r1.x; a1.y += r1.y; a2.x += r2.x; a2.y += r2.y;
    }
    acc[3 * pix] = a0; acc[3 * pix + 1] = a1; acc[3 * pix + 2] = a2;
}

// write_frame_kernel for the AOV sums; albedo / normal may each be null
__global__ void __launch_bounds__(256) aov_write_kernel(const double2* __restrict__ acc, DRender rp, double divisor, double* __restrict__ albedo,
                                                         double* __restrict__ normal) {
    const size_t npix = static_cast<size_t>(rp.tile_w) * rp.tile_h;
    const size_t pix = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (pix >= npix) return;
    const size_t px = frame_pixel(rp, pix);
    const double2 a0 = acc[3 * pix], a1 = acc[3 * pix + 1], a2 = acc[3 * pix + 2];
    double v[6] = {a0.x, a0.y, a1.x, a1.y, a2.x, a2.y};
    if (divisor != 0.0)
        for (int k = 0; k < 6; ++k) v[k] = v[k] / divisor;
    if (albedo) { albedo[3 * px + 0] = v[0]; albedo[3 * px + 1] = v[1]; albedo[3 * px + 2] = v[2]; }
    if (normal) { normal[3 * px + 0] = v[3]; normal[3 * px + 1] = v[4]; normal[3 * px + 2] = v[5]; }
}

// ---------------------------------------------------------------------------------------------
// rtp_render_adaptive (DESIGN.md §6b). Per tile pixel: acc (the colour / foreground sums of resolve_kernel), the luminance
// moments (Σ Y, Σ Y²) and the sample count; per live slot a keep flag. Every sum starts at 0.0 and runs in sample order, so a
// pixel that stops after n samples holds the bits rtp_render's resolve_kernel holds for the sample range [0, n).
// ---------------------------------------------------------------------------------------------

struct StopRule {
    double abs_tol, rel_tol;
    uint32_t max_samples, _pad;
};

__global__ void __launch_bounds__(256) adaptive_init_kernel(double4* __restrict__ acc, double2* __restrict__ moments, uint32_t* __restrict__ count,
                                                            uint32_t* __restrict__ live, size_t npix) {
    const size_t pix = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (pix >= npix) return;
    acc[pix] = make_double4(0.0, 0.0, 0.0, 0.0);
    moments[pix] = make_double2(0.0, 0.0);
    count[pix] = 0u;
    live[pix] = static_cast<uint32_t>(pix);
}

// One launch of a round: for live slot k, the launch's samples of tile pixel live[k] (scratch[k * n_samples + s], path_rng)
// are folded into its sums in sample order. On the round's last launch the stop rule decides keep[k].
__global__ void __launch_bounds__(256) adaptive_resolve_kernel(const double4* __restrict__ scratch, const uint32_t* __restrict__ live, uint32_t n_live,
                                                               uint32_t n_samples, double4* __restrict__ acc, double2* __restrict__ moments,
                                                               uint32_t* __restrict__ count, uint8_t* __restrict__ keep, int last_launch, StopRule rule) {
    const size_t k = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (k >= n_live) return;
    const uint32_t pix = live[k];
    double4 a = acc[pix];
    double2 m = moments[pix];
    for (uint32_t s = 0; s < n_samples; ++s) {
        const double4 c = scratch[k * n_samples + s];
        a.x += c.x; a.y += c.y; a.z += c.z; a.w += c.w;
        const double y = (0.2126 * c.x + 0.7152 * c.y) + 0.0722 * c.z;
        m.x += y; m.y += y * y;
    }
    acc[pix] = a;
    moments[pix] = m;
    const uint32_t n = count[pix] + n_samples;
    count[pix] = n;
    if (last_launch) {
        const double nd = static_cast<double>(n);
        const double mean = m.x / nd;
        const double var = (m.y - m.x * mean) / (nd - 1.0);
        const double tol = rule.abs_tol + rule.rel_tol * fabs(mean);
        const bool stop = n >= rule.max_samples || (n >= 2u && var / nd <= tol * tol);  // NaN / inf: false, the pixel goes on
        keep[k] = stop ? 0 : 1;
    }
}

// write_frame_kernel with each pixel's own divisor: its sample count (no division with RTP_RENDER_RAW_SUMS)
__global__ void __launch_bounds__(256) adaptive_write_kernel(const double4* __restrict__ acc, const uint32_t* __restrict__ count, DRender rp, int raw_sums,
                                                             double* __restrict__ rgb, double* __restrict__ fg, uint32_t* __restrict__ samples) {
    const size_t npix = static_cast<size_t>(rp.tile_w) * rp.tile_h;
    const size_t pix = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (pix >= npix) return;
    const size_t px = frame_pixel(rp, pix);
    double4 a = acc[pix];
    const uint32_t n = count[pix];
    if (!raw_sums) {
        const double divisor = static_cast<double>(n);
        a.x = a.x / divisor; a.y = a.y / divisor; a.z = a.z / divisor; a.w = a.w / divisor;
    }
    rgb[3 * px + 0] = a.x; rgb[3 * px + 1] = a.y; rgb[3 * px + 2] = a.z;
    if (fg) fg[px] = a.w;
    if (samples) samples[px] = n;
}

// Output stage (main.rs:110-122 + utility.rs:212-220 to_srgb_u8): colour = sum / divisor, clamp, gamma 1/2.2, `as u8`;
// alpha = 255, or (255 * foreground) as u8 with RTP_RENDER_TRANSPARENT. CUDA's pow and the host libm's powf may differ in
// the last ulps, which matters only when 255 * x^(1/2.2) lands within 1e-9 of an integer: those pixels (a handful per
// frame at most) are appended to a fix-up list with their f64 colour and redone by the host with its own libm, so the
// bytes are the reference's.
struct SrgbFix {
    uint32_t pixel, _pad;
    double rgb[3];
};

__device__ __forceinline__ uint8_t sat_u8(double y) { return y != y || y <= 0.0 ? 0 : (y >= 255.0 ? 255 : static_cast<uint8_t>(static_cast<int>(y))); }

__global__ void __launch_bounds__(256) srgb8_kernel(const double4* __restrict__ acc, DRender rp, double divisor, int transparent, uchar4* __restrict__ rgba,
                                                     SrgbFix* __restrict__ fixes, unsigned int* __restrict__ n_fixes, unsigned int fix_cap) {
    const size_t npix = static_cast<size_t>(rp.tile_w) * rp.tile_h;
    const size_t pix = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (pix >= npix) return;
    const size_t px = frame_pixel(rp, pix);
    double4 a = acc[pix];
    if (divisor != 0.0) { a.x = a.x / divisor; a.y = a.y / divisor; a.z = a.z / divisor; a.w = a.w / divisor; }
    const double c[3] = {a.x, a.y, a.z};
    uint8_t out[3];
    bool ambiguous = false;
    for (int k = 0; k < 3; ++k) {
        const double x = clampd(c[k], 0.0, 1.0);
        const double y = 255.0 * pow(x, 1.0 / 2.2);
        out[k] = sat_u8(y);
        if (x > 0.0 && x < 1.0 && fabs(y - rint(y)) < 1e-9) ambiguous = true;
    }
    rgba[px] = make_uchar4(out[0], out[1], out[2], transparent ? sat_u8(255.0 * a.w) : 0xff);
    if (ambiguous) {
        const unsigned int slot = atomicAdd(n_fixes, 1u);
        if (slot < fix_cap) {
            fixes[slot].pixel = static_cast<uint32_t>(px);
            fixes[slot].rgb[0] = c[0]; fixes[slot].rgb[1] = c[1]; fixes[slot].rgb[2] = c[2];
        }
    }
}

// ---------------------------------------------------------------------------------------------
// device scene
// ---------------------------------------------------------------------------------------------

constexpr int kPipeDepth = 3;
constexpr size_t kAnyOrderBigScene = 262144;  // leaves from which rtp_scene_info.any_order reports 2 (the kernel is the same)
constexpr unsigned kQueueSlots = 64;
constexpr unsigned kLaunchSlots = 8;

// A per-scene device buffer that grows to the largest size a call has asked of it. It frees its memory when destroyed, on the
// device current then: a DeviceScene is deleted with its own device current (device_scene_free).
template <class T>
struct DevBuf {
    T* ptr = nullptr;
    size_t n = 0;  // elements allocated
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { cudaFree(ptr); }
    void release() { cudaFree(ptr); ptr = nullptr; n = 0; }
    // room for `want` elements; the contents do not survive a reallocation, and a failed one leaves the buffer empty
    int reserve(size_t want) {
        if (n >= want) return RTP_OK;
        release();
        const size_t m = std::max<size_t>(want, 1);
        RTP_CUDA(cudaMalloc(reinterpret_cast<void**>(&ptr), m * sizeof(T)));
        n = m;
        return RTP_OK;
    }
};

struct DeviceScene {
    int device = 0;
    Switches sw;                       // read when the scene was created (scene_create_impl)
    DNode* nodes = nullptr;
    DWide* wide = nullptr;
    size_t n_wide = 0;
    double* wide_boxes = nullptr;
    DWide* free_wide = nullptr;        // order-free culling tree of a big scene (any-order lanes), or nullptr
    size_t n_free_wide = 0;
    double* free_boxes = nullptr;
    size_t stack_bytes = 0;            // dynamic shared memory of the persistent kernels: wide_depth x 128 threads x 4 B
    DPrim* prims = nullptr;
    DAttr* attrs = nullptr;
    DMaterial* materials = nullptr;
    DTexture* textures = nullptr;
    std::vector<uint8_t*> images;
    DSceneView view{};
    uint64_t bytes = 0;

    std::mutex lock;  // serialises calls that use the scratch below
    Counters* counters = nullptr;
    // Per-launch device state of the persistent kernels: a self-rearming work queue and the defer list of trace_any_kernel.
    // Slots are handed out round-robin; each remembers the last launch that used it through an event, and the next user's
    // stream waits on that event first, so two launches in flight on different streams never share a queue or a list.
    struct LaunchSlot {
        WorkQueue* wq = nullptr;
        unsigned long long* defer_count = nullptr;
        DevBuf<uint32_t> defer_idx;
        cudaEvent_t last_use = nullptr;
        cudaStream_t stream = nullptr;  // stream of the last launch that used the slot
        bool used = false;
    };
    LaunchSlot slots[kLaunchSlots];
    std::mutex launch_lock;            // acquire slot + enqueue + record event is one critical section per launch
    unsigned slot_seq = 0;
    WorkQueue* queues = nullptr;       // backing store of the slots' queues and defer counters
    int inorder_blocks = 0, inorder_tail_blocks = 0;  // grids of the in-order kernel (batch / tail mode)
    size_t inorder_stack_bytes = 0;
    int any_blocks = 0;                // grid of trace_any_kernel
    size_t any_stack_bytes = 0;        // its dynamic shared memory: any_cap x 128 threads x 8 B of stacks + 8 KiB of cold lane state
    int any_order = 0;                 // != 0: eligible rays take the any-order walk (RTP_TRAVERSAL); 2 marks a scene of >= 262,144 leaves
    uint32_t any_cap = 0;              // any-order stack entries per lane
    cudaStream_t streams[kPipeDepth] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
    cudaEvent_t render_done = nullptr; // end of the last render enqueued: the next render (any stream) waits for it before it
    bool render_pending = false;       //   touches the per-scene scratch (queues, accumulators, counters)
    std::vector<cudaEvent_t> ev_pool;  // render calls with stats: marks around the traversal launches (trace_ms / shade_ms)
    size_t ev_used = 0;
    size_t last_trace_launches = 1;    // kernels the last launch_trace call queued (2 with the deferred in-order launch)
    size_t pending_launches = 0;       // of the render enqueued last (render_end -> render_finish)
    uint64_t pending_paths = 0;
    DevBuf<rtp_ray> stage_rays[kPipeDepth];  // trace_host's pipeline stages
    DevBuf<rtp_hit_full> stage_hits[kPipeDepth];
    DevBuf<double4> scratch, acc;
    // rtp_render_adaptive, per tile pixel and grown like acc: luminance moments (16 B), sample count (4 B), keep flag (1 B), two live-list entries (8 B): 29 B beside acc's 32.
    // The live count of a round goes through n_live to a pinned word that the host reads.
    DevBuf<double2> moments; DevBuf<uint32_t> counts; DevBuf<uint8_t> keep; DevBuf<uint32_t> live[2];
    DevBuf<uint8_t> select_tmp;  // cub::DeviceSelect::Flagged
    DevBuf<uint32_t> n_live; uint32_t* n_live_host = nullptr;
    // rtp_render_aov: the AovRecords of a launch (3 double2 per path, grown like scratch) and their sums (3 double2 per tile pixel)
    DevBuf<double2> aov_rec, aov_acc;
    // wavefront integrator queues (WaveQueues), grown on demand by wave_reserve for wave_capacity paths per launch and a stack of
    // wave_bounces levels
    DevBuf<rtp_ray> wave_rays[2];
    DevBuf<uint4> wave_state[2];
    DevBuf<WaveHit> wave_hits;
    DevBuf<double2> wave_stack;
    DevBuf<unsigned long long> wave_count;
    size_t wave_capacity = 0;
    uint32_t wave_bounces = 0;
    int shade_blocks = 0;              // grid of wave_shade_kernel
    // memory the integrator's per-launch buffers may take (set at upload from the free HBM). A render call sizes its launches
    // against it with its own max_bounce, and the queues it keeps afterwards hold at most max(this budget, what the call itself
    // needs): growing them to the largest capacity seen AND the deepest stack seen would not (1080p x 16 spp at depth 1, then any
    // frame at depth 128: a 204 GB stack), so wave_reserve then reallocates them for the call alone.
    size_t queue_budget_bytes = size_t(4) << 30;
    DevBuf<double> frame;               // staging planes of the host-buffer render calls (render_host, rtp_render_adaptive)
    DevBuf<uint32_t> frame_samples;     // rtp_render_adaptive's samples_out
    DevBuf<uchar4> frame8;              // RGBA8 output stage
    DevBuf<SrgbFix> fixes; DevBuf<unsigned int> n_fixes;
    unsigned int n_fix_host = 0;       // n_fixes of the last rtp_render_srgb8, copied back with the frame
};

template <class T>
static int upload(const std::vector<T>& v, T** out, uint64_t* bytes) {
    const size_t n = std::max<size_t>(v.size(), 1);
    RTP_CUDA(cudaMalloc(reinterpret_cast<void**>(out), n * sizeof(T)));
    if (!v.empty()) RTP_CUDA(cudaMemcpy(*out, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    *bytes += n * sizeof(T);
    return RTP_OK;
}

void device_scene_free(DeviceScene* ds) {
    if (!ds) return;
    cudaFree(ds->nodes); cudaFree(ds->wide); cudaFree(ds->wide_boxes); cudaFree(ds->free_wide); cudaFree(ds->free_boxes); cudaFree(ds->prims); cudaFree(ds->attrs); cudaFree(ds->materials); cudaFree(ds->textures);
    for (uint8_t* p : ds->images) cudaFree(p);
    cudaFree(ds->counters);
    cudaFree(ds->queues);
    for (DeviceScene::LaunchSlot& sl : ds->slots)
        if (sl.last_use) cudaEventDestroy(sl.last_use);
    for (int k = 0; k < kPipeDepth; ++k)
        if (ds->streams[k]) cudaStreamDestroy(ds->streams[k]);
    if (ds->ev_begin) cudaEventDestroy(ds->ev_begin);
    if (ds->ev_end) cudaEventDestroy(ds->ev_end);
    for (cudaEvent_t ev : ds->ev_pool) cudaEventDestroy(ev);
    if (ds->render_done) cudaEventDestroy(ds->render_done);
    if (ds->n_live_host) cudaFreeHost(ds->n_live_host);
    delete ds;
}

uint64_t device_scene_bytes(const DeviceScene* ds) { return ds ? ds->bytes : 0; }

static int g_device = -1;

static int require_device() {
    if (g_device >= 0) return RTP_OK;
    return rtp_init(0);
}

int ensure_device() { return require_device(); }

static int check_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return set_error(RTP_ERR_CUDA, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                                           " (this library has no CPU fallback)");
    if (device < 0 || device >= n) return set_error(RTP_ERR_INVALID, "device index out of range");
    cudaDeviceProp prop;
    RTP_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return set_error(RTP_ERR_CUDA, std::string("device ") + prop.name + " is not compute capability 10.x; kernels are built for sm_100a only");
    return RTP_OK;
}

int current_device() { return g_device; }

int device_scene_upload(const FlatScene& flat, const Switches& sw, int device, DeviceScene** out) {
    int rc = device < 0 ? require_device() : check_device(device);
    if (rc != RTP_OK) return rc;
    if (device < 0) device = g_device;
    RTP_CUDA(cudaSetDevice(device));
    DeviceScene* ds = new DeviceScene();
    ds->device = device;
    ds->sw = sw;
    auto bail = [&](int code) { device_scene_free(ds); return code; };
    // arrays built on a device (rtp_build.cu) are adopted there and copied peer to peer elsewhere; host-built ones are uploaded
    const bool adopt = flat.dev.valid && flat.dev.device == device && !flat.dev.adopted;  // the replica on the building device takes the arrays over
    auto take = [&](auto** dst, auto* src, size_t count) -> int {
        using T = std::remove_pointer_t<std::remove_pointer_t<decltype(dst)>>;
        const size_t bytes = std::max<size_t>(count, 1) * sizeof(T);
        if (!adopt) {
            RTP_CUDA(cudaMalloc(reinterpret_cast<void**>(dst), bytes));
            if (count) RTP_CUDA(cudaMemcpyPeer(*dst, device, src, flat.dev.device, count * sizeof(T)));
        }
        ds->bytes += bytes;
        return RTP_OK;
    };
    if (adopt) {  // all five at once, so that a failure further down frees each array exactly once (with this DeviceScene)
        ds->nodes = flat.dev.nodes; ds->wide = flat.dev.wide; ds->wide_boxes = flat.dev.wide_boxes; ds->prims = flat.dev.prims; ds->attrs = flat.dev.attrs;
        flat.dev.adopted = true;
    }
    if (flat.dev.valid) {
        if ((rc = take(&ds->nodes, flat.dev.nodes, flat.dev.n_nodes)) != RTP_OK) return bail(rc);
        if ((rc = take(&ds->wide, flat.dev.wide, flat.dev.n_wide)) != RTP_OK) return bail(rc);
        if ((rc = take(&ds->wide_boxes, flat.dev.wide_boxes, flat.dev.n_wide * 24)) != RTP_OK) return bail(rc);
    } else {
    if ((rc = upload(flat.nodes, &ds->nodes, &ds->bytes)) != RTP_OK) return bail(rc);
    if ((rc = upload(flat.wide, &ds->wide, &ds->bytes)) != RTP_OK) return bail(rc);
    if ((rc = upload(flat.wide_boxes, &ds->wide_boxes, &ds->bytes)) != RTP_OK) return bail(rc);
    }
    if (!flat.free_wide.empty()) {
        if ((rc = upload(flat.free_wide, &ds->free_wide, &ds->bytes)) != RTP_OK) return bail(rc);
        if ((rc = upload(flat.free_boxes, &ds->free_boxes, &ds->bytes)) != RTP_OK) return bail(rc);
        ds->n_free_wide = flat.free_wide.size();
    }
    // one stack word per tree level and thread; a tree deeper than 96 levels (degenerate geometry) does not get the f32 walk
    // at all (f32_culling below), so its launches carry no stack
    ds->stack_bytes = static_cast<size_t>(flat.wide_depth <= 96 ? std::max<uint32_t>(flat.wide_depth, 1u) : 1u) * 128 * sizeof(uint32_t);
    // the conservative f32 walk: eligible rays of this scene take it unless RTP_F32_CULLING=0
    const bool f32_culling = sw.f32_culling && flat.root_kind == RTP_ROOT_BVH && flat.boxes_finite && flat.scene_mag <= 1e15 && flat.wide_depth <= 96;
    // every eligible scene takes the any-order walk unless RTP_TRAVERSAL=inorder (measured faster from the 4,969-leaf bunny up); it
    // walks in f32 and indexes nodes as 32-bit float4 offsets. 2 marks a big scene in rtp_scene_info only: every any-order scene
    // runs the same trace_any_kernel
    const bool any_ok = sw.any_order && flat.any_ok && f32_culling && flat.wide_count() < (size_t(1) << 28) && flat.free_wide.size() < (size_t(1) << 28);
    ds->any_order = any_ok ? (flat.prim_count() >= kAnyOrderBigScene ? 2 : 1) : 0;
    if (flat.dev.valid) {
        if ((rc = take(&ds->prims, flat.dev.prims, flat.dev.n_prims)) != RTP_OK) return bail(rc);
        if ((rc = take(&ds->attrs, flat.dev.attrs, flat.dev.n_prims)) != RTP_OK) return bail(rc);
    } else {
    if ((rc = upload(flat.prims, &ds->prims, &ds->bytes)) != RTP_OK) return bail(rc);
    if ((rc = upload(flat.attrs, &ds->attrs, &ds->bytes)) != RTP_OK) return bail(rc);
    }
    if ((rc = upload(flat.materials, &ds->materials, &ds->bytes)) != RTP_OK) return bail(rc);
    std::vector<DTexture> tex = flat.textures;
    ds->images.assign(tex.size(), nullptr);
    for (size_t i = 0; i < tex.size(); ++i) {
        if (flat.images[i].empty()) continue;
        cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&ds->images[i]), flat.images[i].size());
        if (e == cudaSuccess) e = cudaMemcpy(ds->images[i], flat.images[i].data(), flat.images[i].size(), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) return bail(set_error(RTP_ERR_CUDA, std::string("texture upload: ") + cudaGetErrorString(e)));
        tex[i].rgba = ds->images[i];
        ds->bytes += flat.images[i].size();
    }
    if ((rc = upload(tex, &ds->textures, &ds->bytes)) != RTP_OK) return bail(rc);
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&ds->counters), sizeof(Counters));
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&ds->queues), kQueueSlots * sizeof(WorkQueue));
    if (e == cudaSuccess) e = cudaMemset(ds->queues, 0, kQueueSlots * sizeof(WorkQueue));
    for (unsigned k = 0; k < kLaunchSlots && e == cudaSuccess; ++k) {
        // queue entry 2k: the slot's work queue; entry 2k + 1: its defer counter (first 8 bytes)
        ds->slots[k].wq = ds->queues + 2 * k;
        ds->slots[k].defer_count = reinterpret_cast<unsigned long long*>(ds->queues + 2 * k + 1);
        e = cudaEventCreateWithFlags(&ds->slots[k].last_use, cudaEventDisableTiming);
    }
    if (e == cudaSuccess) {
        cudaDeviceProp prop;
        e = cudaGetDeviceProperties(&prop, ds->device);
        int per_sm = 0, tail_per_sm = 0, any_per_sm = 0;
        // in-order kernel (every scene: List roots, scenes outside the any-order walk's preconditions, the rays trace_any_kernel
        // defers, tail-mode launches): one stack word per tree level and thread
        ds->inorder_stack_bytes = ds->stack_bytes;
        if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, trace_persistent_kernel<false, OUT_HIT, false>, 128, ds->inorder_stack_bytes);
        if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&tail_per_sm, trace_persistent_kernel<false, OUT_TAIL, false>, 128, ds->inorder_stack_bytes);
        ds->inorder_blocks = prop.multiProcessorCount * std::max(per_sm, 1);
        ds->inorder_tail_blocks = prop.multiProcessorCount * std::max(tail_per_sm, 1);
        if (ds->any_order) {
            // any-order lanes postpone up to three siblings per level, each with its entry distance (8 B): a primary ray of the bunny
            // never holds more than 16 entries (gpurun_out/r2_sweep1.log: 0 overflows of 2 M rays at 16, 65 of 4 Mi incoherent ones; 1 at 20, 0 at
            // 22 - and ONE deferred ray costs a 20 us second launch, 2 % of that batch),
            // deep trees get up to 28 (a primary ray of the 2.5 M-leaf bunny field runs 4 % FASTER at 24 than at 32: occupancy, not
            // overflows, is what the cap costs); a lane that would need more defers its ray to the in-order kernel
            const uint32_t any_depth = ds->free_wide ? flat.free_depth : flat.wide_depth;
            ds->any_cap = std::max<uint32_t>(4u, std::min<uint32_t>(3u * any_depth + 1u, any_depth <= 12 ? 22u : 28u));  // six blocks per SM: 22 + 8 KiB stay inside the 196 KiB carve-out, 28 + 8 KiB inside 228
            if (sw.any_cap) ds->any_cap = sw.any_cap;  // tests
            ds->any_stack_bytes = static_cast<size_t>(ds->any_cap) * 128 * sizeof(uint2) + kAnyColdBytes;  // the stacks, then the cold state
            if (ds->any_stack_bytes > 48u * 1024u) {  // deep trees: above the default limit of dynamic shared memory, every instantiation that is launched
#define RTP_ANY_SMEM(C, O) if (e == cudaSuccess) e = cudaFuncSetAttribute(trace_any_kernel<C, O>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(ds->any_stack_bytes))
                RTP_ANY_SMEM(false, OUT_HIT); RTP_ANY_SMEM(true, OUT_HIT); RTP_ANY_SMEM(false, OUT_FULL); RTP_ANY_SMEM(true, OUT_FULL);
                RTP_ANY_SMEM(false, OUT_WAVE); RTP_ANY_SMEM(true, OUT_WAVE);
#undef RTP_ANY_SMEM
            }
            if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&any_per_sm, trace_any_kernel<false, OUT_HIT>, 128, ds->any_stack_bytes);
            ds->any_blocks = prop.multiProcessorCount * std::max(any_per_sm, 1);
        }
        size_t free_b = 0, total_b = 0;
        if (e == cudaSuccess && cudaMemGetInfo(&free_b, &total_b) == cudaSuccess)
            ds->queue_budget_bytes = std::max<size_t>(size_t(1) << 30, std::min<size_t>(size_t(24) << 30, free_b / 6));
        ds->shade_blocks = prop.multiProcessorCount * kShadeBlocks;
        if (sw.build_timing)
            std::fprintf(stderr, "[rtp build] 4-wide tree depth %u (order-free tree: %u), %s walk (%u big primitives), %zu B of stack per block, %d traversal blocks per SM\n",
                         flat.wide_depth, flat.free_depth, ds->any_order ? "any-order" : "in-order", flat.n_big,
                         ds->any_order ? ds->any_stack_bytes : ds->stack_bytes, ds->any_order ? any_per_sm : per_sm);
    }
    for (int k = 0; k < kPipeDepth && e == cudaSuccess; ++k) e = cudaStreamCreateWithFlags(&ds->streams[k], cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&ds->ev_begin);
    if (e == cudaSuccess) e = cudaEventCreate(&ds->ev_end);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ds->render_done, cudaEventDisableTiming);
    if (e != cudaSuccess) return bail(set_error(RTP_ERR_CUDA, std::string("scene resources: ") + cudaGetErrorString(e)));

    ds->n_wide = flat.wide_count();
    DSceneView& v = ds->view;
    v.nodes = ds->nodes; v.wide = ds->wide; v.wide_boxes = ds->wide_boxes; v.prims = ds->prims;
    v.any_wide = ds->free_wide ? ds->free_wide : ds->wide; v.any_boxes = ds->free_wide ? ds->free_boxes : ds->wide_boxes;
    v.f32_culling = f32_culling ? 1u : 0u; v.attrs = ds->attrs; v.materials = ds->materials; v.textures = ds->textures;
    v.n_nodes = flat.root_kind == RTP_ROOT_BVH ? static_cast<uint32_t>(flat.node_count()) : 0u;
    v.n_prims = static_cast<uint32_t>(flat.prim_count());
    v.root_kind = flat.root_kind;
    v.bg_kind = flat.background.kind; v.bg_texture = flat.background.texture;
    v.any_order = ds->any_order ? 1u : 0u;
    v.any_cap = ds->any_cap;
    v.n_big = flat.n_big;
    v.fast_slab = flat.boxes_finite ? 1u : 0u;
    for (int k = 0; k < 8; ++k) v.big[k] = flat.big[k];
    v.any_E = flat.any_E; v.any_A = flat.any_A;
    v.any_Ef = std::nextafter(static_cast<float>(flat.any_E), std::numeric_limits<float>::infinity());  // >= any_E
    v.any_Af = std::nextafter(static_cast<float>(flat.any_A), std::numeric_limits<float>::infinity());
    v.any_Cf = std::nextafter(static_cast<float>(flat.any_C), std::numeric_limits<float>::infinity());
    v.any_Rf = flat.any_spheres ? std::nextafter(static_cast<float>(flat.any_R), std::numeric_limits<float>::infinity()) : -1.0f;
    std::memcpy(v.bg_rgb, flat.background.rgb, sizeof v.bg_rgb);
    // RTP_ANY_SETUP_CULL=0: a box that every ray enters, so every ray walks (A/B runs of the set-up cull in one process)
    for (int k = 0; k < 6; ++k) v.cull[k] = sw.any_setup_cull ? flat.cull[k] : (k < 3 ? -1.0f : 1.0f) * std::numeric_limits<float>::infinity();
    *out = ds;
    return RTP_OK;
}

static DCamera make_camera(const rtp_camera* c) {
    DCamera d;
    d.tan_fov = std::tan(0.5 * c->fov);  // render.rs:33, evaluated by the host libm like the reference
    d.focal_dist = c->focal_dist; d.aspect_ratio = c->aspect_ratio; d.lens_radius = c->lens_radius;
    std::memcpy(d.m, c->orientation, sizeof d.m);
    std::memcpy(d.pos, c->position, sizeof d.pos);
    return d;
}

// One traversal launch. out_mode: OUT_HIT / OUT_FULL / OUT_WAVE / OUT_TAIL / OUT_OCCLUDED. n_dev != nullptr: the batch size is read from device memory
// (wavefront integrator) and `n` is only an upper bound used to size the grid.
// RTP_DEBUG_SYNC=1: synchronise after every launch of the integrator and name the kernel that faulted
static int debug_sync(const DeviceScene* ds, cudaStream_t st, const char* what, uint32_t bounce) {
    if (!ds->sw.debug_sync) return RTP_OK;
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return set_error(RTP_ERR_CUDA, std::string(what) + " (segment " + std::to_string(bounce) + "): " + cudaGetErrorString(e));
    return RTP_OK;
}

static int launch_trace(DeviceScene* ds, const rtp_ray* d_rays, size_t n, void* d_out, int out_mode, bool count, Counters* counters,
                        cudaStream_t stream, const unsigned long long* n_dev = nullptr, const TailArgs* tail = nullptr) {
    if (n == 0) return RTP_OK;
    const unsigned block = 128;
    ds->last_trace_launches = 1;
    if (ds->sw.simple_trace && !n_dev && out_mode != OUT_WAVE) {
        const size_t grid = (n + block - 1) / block;
        if (grid > 0x7FFFFFFFull) return set_error(RTP_ERR_INVALID, "ray batch too large for one launch");
        const dim3 g(static_cast<unsigned>(grid));
        if (out_mode == OUT_FULL) {
            if (count) trace_closest_kernel<true, true><<<g, block, 0, stream>>>(ds->view, d_rays, n, d_out, counters);
            else trace_closest_kernel<false, true><<<g, block, 0, stream>>>(ds->view, d_rays, n, d_out, counters);
        } else if (out_mode == OUT_OCCLUDED) {
            if (count) trace_occluded_simple_kernel<true><<<g, block, 0, stream>>>(ds->view, d_rays, n, d_out, counters);
            else trace_occluded_simple_kernel<false><<<g, block, 0, stream>>>(ds->view, d_rays, n, d_out, counters);
        } else {
            if (count) trace_closest_kernel<true, false><<<g, block, 0, stream>>>(ds->view, d_rays, n, d_out, counters);
            else trace_closest_kernel<false, false><<<g, block, 0, stream>>>(ds->view, d_rays, n, d_out, counters);
        }
    } else {
        // persistent grid: a whole number of resident blocks per SM, never more warps than rays
        const size_t want = (n + 3) / 4;  // a warp per ray at least: small batches are latency-bound per warp, so they are spread thin
        const bool list = ds->view.root_kind != RTP_ROOT_BVH;
        const TailArgs ta = tail ? *tail : TailArgs{};
        // which kernel: the any-order kernel + a deferred in-order launch (eligible scenes), or the in-order kernel alone (List roots,
        // scenes outside the preconditions, tail-mode launches, occlusion queries: with T fixed the walk order does not matter)
        const bool pure_any = !list && ds->any_order && out_mode != OUT_TAIL && out_mode != OUT_OCCLUDED;
        if (n > 0xFFFFFFFEull && pure_any) return set_error(RTP_ERR_INVALID, "ray batch too large for one launch");

        std::lock_guard<std::mutex> guard(ds->launch_lock);
        // a stream keeps its slot (launches on one stream are ordered anyway, and the slot's defer list is already sized);
        // a new stream takes an unused slot, or the next one round-robin after waiting for that slot's last launch
        DeviceScene::LaunchSlot* pick = nullptr;
        for (DeviceScene::LaunchSlot& sl : ds->slots)
            if (sl.used && sl.stream == stream) { pick = &sl; break; }
        if (!pick)
            for (DeviceScene::LaunchSlot& sl : ds->slots)
                if (!sl.used) { pick = &sl; break; }
        if (!pick) {
            pick = &ds->slots[ds->slot_seq++ % kLaunchSlots];
            RTP_CUDA(cudaStreamWaitEvent(stream, pick->last_use, 0));  // its previous launch, on another stream, must be over
        }
        DeviceScene::LaunchSlot& slot = *pick;
        if (pure_any && slot.defer_idx.n < n) {
            if (slot.used) RTP_CUDA(cudaEventSynchronize(slot.last_use));  // its last launch may still read the list
            if (int rc = slot.defer_idx.reserve(std::max<size_t>(n, 65536))) return rc;
        }
        WorkQueue* wq = slot.wq;
        const DeferList no_index{nullptr, nullptr};
        if (pure_any) {
            const dim3 g(static_cast<unsigned>(std::min<size_t>(static_cast<size_t>(ds->any_blocks), want)));
            const DeferList defer{slot.defer_idx.ptr, slot.defer_count};
#define RTP_LAUNCH_ANY(C, O) trace_any_kernel<C, O><<<g, block, ds->any_stack_bytes, stream>>>(ds->view, d_rays, n, d_out, counters, wq, n_dev, defer)
            if (out_mode == OUT_FULL) { if (count) RTP_LAUNCH_ANY(true, OUT_FULL); else RTP_LAUNCH_ANY(false, OUT_FULL); }
            else if (out_mode == OUT_WAVE) { if (count) RTP_LAUNCH_ANY(true, OUT_WAVE); else RTP_LAUNCH_ANY(false, OUT_WAVE); }
            else { if (count) RTP_LAUNCH_ANY(true, OUT_HIT); else RTP_LAUNCH_ANY(false, OUT_HIT); }
#undef RTP_LAUNCH_ANY
            RTP_CUDA(cudaGetLastError());
            if (out_mode == OUT_WAVE) {
                // inside the integrator the (rare) rays this kernel does not answer are traced by the thread that shades them
                RTP_CUDA(cudaEventRecord(slot.last_use, stream));
                slot.used = true;
                slot.stream = stream;
                return RTP_OK;
            }
            // the deferred rays (normally none: the launch then finds an empty list and leaves at once), in the reference's order
            const dim3 g2(static_cast<unsigned>(std::min<size_t>(static_cast<size_t>(ds->inorder_blocks), want)));
            // programmatic dependent launch: the launch latency of this (normally empty) pass hides behind the tail of trace_any_kernel
            cudaLaunchAttribute pdl;
            pdl.id = cudaLaunchAttributeProgrammaticStreamSerialization;
            pdl.val.programmaticStreamSerializationAllowed = 1;
            cudaLaunchConfig_t cfg2 = {};
            cfg2.gridDim = g2; cfg2.blockDim = block; cfg2.dynamicSmemBytes = ds->inorder_stack_bytes; cfg2.stream = stream;
            cfg2.attrs = &pdl; cfg2.numAttrs = 1;
            const unsigned long long* const no_n_dev = nullptr;
#define RTP_LAUNCH_DEFERRED(C, O) RTP_CUDA(cudaLaunchKernelEx(&cfg2, trace_persistent_kernel<C, O, false>, ds->view, d_rays, n, d_out, counters, wq, no_n_dev, ta, defer))
            if (out_mode == OUT_FULL) { if (count) RTP_LAUNCH_DEFERRED(true, OUT_FULL); else RTP_LAUNCH_DEFERRED(false, OUT_FULL); }
            else if (out_mode == OUT_WAVE) { if (count) RTP_LAUNCH_DEFERRED(true, OUT_WAVE); else RTP_LAUNCH_DEFERRED(false, OUT_WAVE); }
            else { if (count) RTP_LAUNCH_DEFERRED(true, OUT_HIT); else RTP_LAUNCH_DEFERRED(false, OUT_HIT); }
#undef RTP_LAUNCH_DEFERRED
            ds->last_trace_launches = 2;
        } else {
            const int blocks = out_mode == OUT_TAIL ? ds->inorder_tail_blocks : ds->inorder_blocks;
            const size_t smem = ds->inorder_stack_bytes;
            const dim3 g(static_cast<unsigned>(std::min<size_t>(static_cast<size_t>(blocks), want)));
#define RTP_LAUNCH_PERSISTENT(C, O, L) trace_persistent_kernel<C, O, L><<<g, block, smem, stream>>>(ds->view, d_rays, n, d_out, counters, wq, n_dev, ta, no_index)
#define RTP_LAUNCH_PERSISTENT_O(O)                                                                   \
    do {                                                                                             \
        if (list) { if (count) RTP_LAUNCH_PERSISTENT(true, O, true); else RTP_LAUNCH_PERSISTENT(false, O, true); }     \
        else { if (count) RTP_LAUNCH_PERSISTENT(true, O, false); else RTP_LAUNCH_PERSISTENT(false, O, false); }        \
    } while (0)
            if (out_mode == OUT_FULL) RTP_LAUNCH_PERSISTENT_O(OUT_FULL);
            else if (out_mode == OUT_WAVE) RTP_LAUNCH_PERSISTENT_O(OUT_WAVE);
            else if (out_mode == OUT_TAIL) RTP_LAUNCH_PERSISTENT_O(OUT_TAIL);
            else if (out_mode == OUT_OCCLUDED) RTP_LAUNCH_PERSISTENT_O(OUT_OCCLUDED);
            else RTP_LAUNCH_PERSISTENT_O(OUT_HIT);
#undef RTP_LAUNCH_PERSISTENT_O
#undef RTP_LAUNCH_PERSISTENT
        }
        RTP_CUDA(cudaGetLastError());
        RTP_CUDA(cudaEventRecord(slot.last_use, stream));
        slot.used = true;
        slot.stream = stream;
        return RTP_OK;
    }
    RTP_CUDA(cudaGetLastError());
    return RTP_OK;
}

// The scene's counters and the ev_begin -> ev_end time of the finished call that used them last, as the rtp_stats fields they give
// (every other field 0). c != nullptr: the raw counters too.
static int read_stats(const DeviceScene* ds, rtp_stats* stats, Counters* c = nullptr) {
    Counters local;
    if (!c) c = &local;
    RTP_CUDA(cudaMemcpy(c, ds->counters, sizeof *c, cudaMemcpyDeviceToHost));
    float ms = 0.f;
    RTP_CUDA(cudaEventElapsedTime(&ms, ds->ev_begin, ds->ev_end));
    std::memset(stats, 0, sizeof *stats);
    stats->rays = c->rays; stats->node_visits = c->node_visits; stats->triangle_tests = c->triangle_tests; stats->sphere_tests = c->sphere_tests;
    stats->leaf_gates = c->leaf_gates; stats->conservative_violations = c->violations; stats->order_rewalks = c->rewalks;
    stats->device_ms = ms;
    return RTP_OK;
}

static void add_stats(rtp_stats* total, const rtp_stats& one) {
    total->rays += one.rays; total->paths += one.paths; total->node_visits += one.node_visits; total->triangle_tests += one.triangle_tests;
    total->sphere_tests += one.sphere_tests; total->leaf_gates += one.leaf_gates; total->conservative_violations += one.conservative_violations;
    total->order_rewalks += one.order_rewalks; total->kernel_launches += one.kernel_launches;
    total->device_ms = std::max(total->device_ms, one.device_ms);  // the devices run side by side
    total->trace_ms = std::max(total->trace_ms, one.trace_ms); total->shade_ms = std::max(total->shade_ms, one.shade_ms);
}

// Host-buffer batch: chunks flow H2D → kernel → D2H on kPipeDepth streams per device so copies overlap traversal; a scene that
// lives on several devices (rtp_scene_create_multi) deals its chunks out to them round-robin, so every device's host link carries
// a share of the 80 B/ray stream. Chunks are independent: no exchange between devices.
// `camera` != nullptr: the rays are pixel-centre camera rays generated on the device chunk by chunk (rtp_trace_camera)
// out_mode: OUT_HIT (16 B rtp_hit), OUT_FULL (80 B rtp_hit_full) or OUT_OCCLUDED (1 B) records
static int trace_host(rtp_scene* scene, const rtp_ray* rays, size_t n, void* hits_out, int out_mode, rtp_stats* stats, const DCamera* camera = nullptr,
                      uint32_t width = 0, uint32_t height = 0) {
    const std::vector<DeviceScene*>& devs = scene->devs;
    const size_t N = devs.size();
    std::vector<std::unique_lock<std::mutex>> locks;
    for (DeviceScene* ds : devs) locks.emplace_back(ds->lock);
    const size_t hit_bytes = out_mode == OUT_FULL ? sizeof(rtp_hit_full) : out_mode == OUT_OCCLUDED ? sizeof(uint8_t) : sizeof(rtp_hit);
    const bool count = stats != nullptr;
    const size_t chunk = size_t(1) << devs[0]->sw.chunk_log2;  // rays per pipeline stage: 2^18 (16 MiB of rays) unless RTP_CHUNK_LOG2 says otherwise
    const size_t n_chunks = (n + chunk - 1) / chunk;
    const size_t used = std::min(N, n_chunks);  // devices that get at least one chunk
    int rc = RTP_OK;
    for (size_t d = 0; d < used && rc == RTP_OK; ++d) {
        DeviceScene* ds = devs[d];
        RTP_CUDA(cudaSetDevice(ds->device));
        for (int k = 0; k < kPipeDepth; ++k) {
            if ((rc = ds->stage_rays[k].reserve(chunk)) != RTP_OK) return rc;
            if ((rc = ds->stage_hits[k].reserve(chunk)) != RTP_OK) return rc;
        }
        if (count) RTP_CUDA(cudaMemsetAsync(ds->counters, 0, sizeof(Counters), ds->streams[0]));
        RTP_CUDA(cudaEventRecord(ds->ev_begin, ds->streams[0]));
        for (int k = 1; k < kPipeDepth; ++k) RTP_CUDA(cudaStreamWaitEvent(ds->streams[k], ds->ev_begin, 0));
    }
    size_t launches = 0, chunk_id = 0;
    for (size_t off = 0; off < n && rc == RTP_OK; off += chunk, ++chunk_id) {
        const size_t m = std::min(chunk, n - off);
        DeviceScene* ds = devs[chunk_id % N];
        const int k = static_cast<int>((chunk_id / N) % kPipeDepth);
        cudaStream_t st = ds->streams[k];
        cudaError_t e = N > 1 ? cudaSetDevice(ds->device) : cudaSuccess;
        if (e == cudaSuccess) {
            if (camera) {
                camera_rays_kernel<<<static_cast<unsigned>((m + 255) / 256), 256, 0, st>>>(*camera, width, height, ds->stage_rays[k].ptr, off, m);
                e = cudaGetLastError();
                ++launches;
            } else {
                e = cudaMemcpyAsync(ds->stage_rays[k].ptr, rays + off, m * sizeof(rtp_ray), cudaMemcpyHostToDevice, st);
            }
        }
        if (e != cudaSuccess) { rc = set_error(RTP_ERR_CUDA, std::string("trace chunk: ") + cudaGetErrorString(e)); break; }
        rc = launch_trace(ds, ds->stage_rays[k].ptr, m, ds->stage_hits[k].ptr, out_mode, false, count ? ds->counters : nullptr, st);
        if (rc != RTP_OK) break;
        launches += ds->last_trace_launches;
        e = cudaMemcpyAsync(static_cast<char*>(hits_out) + off * hit_bytes, ds->stage_hits[k].ptr, m * hit_bytes, cudaMemcpyDeviceToHost, st);
        if (e != cudaSuccess) rc = set_error(RTP_ERR_CUDA, std::string("trace chunk: ") + cudaGetErrorString(e));
    }
    // drain every device that was given work (also after an error: nothing may stay in flight on the staging buffers)
    rtp_stats total;
    std::memset(&total, 0, sizeof total);
    for (size_t d = 0; d < used; ++d) {
        DeviceScene* ds = devs[d];
        cudaSetDevice(ds->device);
        cudaError_t e = cudaSuccess;
        for (int k = 1; k < kPipeDepth && e == cudaSuccess; ++k) e = cudaStreamSynchronize(ds->streams[k]);
        if (e == cudaSuccess) e = cudaEventRecord(ds->ev_end, ds->streams[0]);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ds->streams[0]);
        else cudaStreamSynchronize(ds->streams[0]);
        if (e != cudaSuccess && rc == RTP_OK) rc = set_error(RTP_ERR_CUDA, std::string("trace: ") + cudaGetErrorString(e));
        if (stats && rc == RTP_OK) {
            rtp_stats one;
            if ((rc = read_stats(ds, &one)) == RTP_OK) add_stats(&total, one);
        }
    }
    if (N > 1) cudaSetDevice(scene->dev->device);
    if (stats && rc == RTP_OK) { total.kernel_launches = launches; *stats = total; }
    return rc;
}

template <int MAXB, class Map, class Aov>
static void launch_render_paths(DeviceScene* ds, const DCamera& cam, const DRender& rp, const Map& map, const Aov& aov, size_t total, bool count,
                                cudaStream_t st) {
    const unsigned block = 128;
    const dim3 g(static_cast<unsigned>((total + block - 1) / block));
    if (count) render_paths_kernel<MAXB, true><<<g, block, 0, st>>>(ds->view, cam, rp, ds->scratch.ptr, ds->counters, map, aov);
    else render_paths_kernel<MAXB, false><<<g, block, 0, st>>>(ds->view, cam, rp, ds->scratch.ptr, ds->counters, map, aov);
}

// bytes per path of one launch of the wavefront integrator: what wave_reserve allocates per path (two queue rays and states, a hit
// record, `bounces` levels of the [bounce][path] stack: 192 B + 48 B per level) and the path's scratch entry (32 B)
static size_t wave_path_bytes(uint32_t bounces) {
    return 2 * (sizeof(rtp_ray) + sizeof(uint4)) + sizeof(WaveHit) + WaveQueues::kLevel * sizeof(double2) * bounces + sizeof(double4);
}

constexpr size_t kWaveCounts = kMaxBounce + 2;  // count[b] for b <= kMaxBounce, and one spare

// Sizes the wavefront queues for `capacity` paths per launch and a stack of `bounces` levels. The queues grow to cover every
// shape seen so far, unless that union would cross queue_budget_bytes: then they are sized for this call alone (see
// DeviceScene::queue_budget_bytes), and the larger ones are let go first.
static int wave_reserve(DeviceScene* ds, size_t capacity, uint32_t bounces) {
    if (ds->wave_capacity >= capacity && ds->wave_bounces >= bounces) return RTP_OK;
    const size_t grown_cap = std::max(capacity, ds->wave_capacity);
    const uint32_t grown_bounces = std::max(bounces, ds->wave_bounces);
    if (grown_cap * wave_path_bytes(grown_bounces) <= std::max(ds->queue_budget_bytes, capacity * wave_path_bytes(bounces))) {
        capacity = grown_cap;
        bounces = grown_bounces;
    } else {
        for (int k = 0; k < 2; ++k) { ds->wave_rays[k].release(); ds->wave_state[k].release(); }
        ds->wave_hits.release(); ds->wave_stack.release();
    }
    ds->wave_capacity = 0;
    ds->wave_bounces = 0;
    for (int k = 0; k < 2; ++k) {
        if (int rc = ds->wave_rays[k].reserve(capacity)) return rc;
        if (int rc = ds->wave_state[k].reserve(capacity)) return rc;
    }
    if (int rc = ds->wave_hits.reserve(capacity)) return rc;
    if (int rc = ds->wave_stack.reserve(capacity * bounces * WaveQueues::kLevel)) return rc;
    if (int rc = ds->wave_count.reserve(kWaveCounts)) return rc;
    ds->wave_capacity = capacity;
    ds->wave_bounces = bounces;
    return RTP_OK;
}

// the queues as the integrator kernels take them
static WaveQueues wave_queues(const DeviceScene* ds) {
    return WaveQueues{{ds->wave_rays[0].ptr, ds->wave_rays[1].ptr}, {ds->wave_state[0].ptr, ds->wave_state[1].ptr}, ds->wave_hits.ptr,
                      ds->wave_stack.ptr, ds->wave_count.ptr, ds->wave_capacity};
}

constexpr unsigned int kSrgbFixCap = 1u << 16;

// d_rgba8 != nullptr: the output stage runs on the device (srgb8_kernel) instead of write_frame_kernel.
// Two phases so that one host thread can keep several devices busy: render_enqueue queues every launch of the frame on `st`
// without synchronising, render_finish waits for them and reads the counters back.
static cudaEvent_t next_mark(DeviceScene* ds, cudaStream_t st) {
    if (ds->ev_used == ds->ev_pool.size()) {
        cudaEvent_t ev = nullptr;
        if (cudaEventCreate(&ev) != cudaSuccess) return nullptr;
        ds->ev_pool.push_back(ev);
    }
    cudaEvent_t ev = ds->ev_pool[ds->ev_used++];
    cudaEventRecord(ev, st);
    return ev;
}

// The pixels a render call covers: checks the frame, tile and row parameters shared by rtp_render and rtp_render_adaptive and
// returns the DRender of the call (tile_h = rows of the tile rectangle this call renders; sample range still unset).
// fixed_spp: rtp_render's sample range is checked too (rtp_render_adaptive checks its own).
static int render_rect(const rtp_render_params* p, bool fixed_spp, DRender* rp) {
    if (p->max_bounce < 1) return set_error(RTP_ERR_INVALID, "assert!(depth >= 1) (render.rs:97)");
    if (p->max_bounce > kMaxBounce) return set_error(RTP_ERR_UNSUPPORTED, "max_bounce > 128");
    if (p->width == 0 || p->height == 0 || (fixed_spp && (p->sample_end < p->sample_begin || p->num_samples == 0)))
        return set_error(RTP_ERR_INVALID, "bad frame parameters");
    if (static_cast<uint64_t>(p->width) * p->height > 0xFFFFFFFFull) return set_error(RTP_ERR_INVALID, "frame too large");
    const uint32_t tx = p->tile_x, ty = p->tile_y;
    if (tx >= p->width || ty >= p->height) return set_error(RTP_ERR_INVALID, "tile outside frame");
    const uint32_t tw = p->tile_w ? p->tile_w : p->width - tx, th_full = p->tile_h ? p->tile_h : p->height - ty;
    if (static_cast<uint64_t>(tx) + tw > p->width || static_cast<uint64_t>(ty) + th_full > p->height) return set_error(RTP_ERR_INVALID, "tile outside frame");
    const uint32_t rs = p->row_stride ? p->row_stride : 1u, ro = p->row_offset;
    if (ro >= rs) return set_error(RTP_ERR_INVALID, "row_offset must be below row_stride");
    const uint32_t th = ro < th_full ? (th_full - ro + rs - 1u) / rs : 0u;  // rows of the tile rectangle this call renders
    rp->width = p->width; rp->height = p->height; rp->max_bounce = p->max_bounce;
    rp->tile_x = tx; rp->tile_y = ty; rp->tile_w = tw; rp->tile_h = th;
    rp->row_offset = ro; rp->row_stride = rs;
    rp->sample_begin = 0; rp->n_samples = 0;
    rp->_pad = 0; rp->seed = p->seed;
    return RTP_OK;
}

// Takes the scene's render scratch (integrator queues, accumulators, counters, time marks) for a call on `st`: checks the call's
// pixels (render_rect), orders `st` after the render queued last on any stream, zeroes the counters and opens the timed span.
// On RTP_OK the call holds the scratch until render_end, which it runs after an error too.
static int render_begin(DeviceScene* ds, const rtp_render_params* p, bool fixed_spp, bool want_stats, cudaStream_t st, DRender* rp) {
    if (int rc = render_rect(p, fixed_spp, rp)) return rc;
    if (ds->render_pending) RTP_CUDA(cudaStreamWaitEvent(st, ds->render_done, 0));
    ds->ev_used = 0;
    RTP_CUDA(cudaMemsetAsync(ds->counters, 0, sizeof(Counters), st));
    if (want_stats) {
        RTP_CUDA(cudaEventRecord(ds->ev_begin, st));
        RTP_CUDA(cudaEventRecord(ds->ev_end, st));
    }
    return RTP_OK;
}

// Releases the scratch after the call's last launch on `st`: keeps its kernel and path counts for render_finish, closes the timed
// span and records render_done, which the next render waits for before it touches the scratch, also when this call failed part way.
static int render_end(DeviceScene* ds, cudaStream_t st, bool want_stats, size_t launches, uint64_t paths) {
    ds->pending_launches = launches;
    ds->pending_paths = paths;
    if (want_stats) RTP_CUDA(cudaEventRecord(ds->ev_end, st));
    RTP_CUDA(cudaEventRecord(ds->render_done, st));
    ds->render_pending = true;
    return RTP_OK;
}

// Paths per launch of the integrator for a call with max_bounce `bounces`: up to 32 Mi paths (wave_path_bytes per path), within
// the memory budget fixed when the scene was uploaded (a sixth of the free HBM, at most 24 GiB). Big launches matter: every launch
// pays the fill and drain of ~2 x max_bounce kernels and the latency-bound sparse late bounces once (1080p x 64 spp of the C4
// scene: 111 ms in 16 launches of 8 Mi paths, 92 ms in 4 launches of 32 Mi). An AOV call (rtp_render_aov) adds its 48-byte
// AovRecords per path.
static size_t path_budget(const DeviceScene* ds, uint32_t bounces, bool aov = false) {
    const size_t per_path = (ds->sw.simple_render ? 32 : wave_path_bytes(bounces)) + (aov ? 3 * sizeof(double2) : 0);
    size_t budget = std::max<size_t>(size_t(1) << 20, std::min<size_t>(size_t(32) << 20, ds->queue_budget_bytes / per_path));
    if (const size_t forced = read_path_budget()) budget = forced;  // tests: force several launches per frame
    return budget;
}

// the integrator's per-launch buffers for launches of up to `need` paths (aov: with their AovRecords)
static int reserve_paths(DeviceScene* ds, size_t need, uint32_t bounces, bool aov = false) {
    if (!ds->sw.simple_render) {
        int rc = wave_reserve(ds, need, bounces);
        if (rc != RTP_OK) return rc;
    }
    if (int rc = ds->scratch.reserve(need)) return rc;
    return aov ? ds->aov_rec.reserve(need * 3) : RTP_OK;
}

// One launch of the integrator: the `total` paths of rp's sample range over the pixel slots of `map`, traced to their end; path p's
// colour and foreground land in ds->scratch[p], and with AovRecords its first vertex in aov.rec[3 p ...]. Adds the kernels it queued
// to *launches.
template <class Map, class Aov>
static int launch_paths(DeviceScene* ds, const DCamera& cam, const DRender& rp, const Map& map, const Aov& aov, size_t total, bool count,
                        bool want_stats, cudaStream_t st, size_t* launches) {
    if (ds->sw.simple_render) {
        if (rp.max_bounce <= 8) launch_render_paths<8>(ds, cam, rp, map, aov, total, count, st);
        else if (rp.max_bounce <= 32) launch_render_paths<32>(ds, cam, rp, map, aov, total, count, st);
        else launch_render_paths<kMaxBounce>(ds, cam, rp, map, aov, total, count, st);
        RTP_CUDA(cudaGetLastError());
        ++*launches;
        return RTP_OK;
    }
    // generate -> (trace -> shade) x max_bounce; queue sizes stay on the device
    const WaveQueues wq = wave_queues(ds);
    RTP_CUDA(cudaMemsetAsync(wq.count, 0, kWaveCounts * sizeof(unsigned long long), st));
    wave_generate_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, st>>>(cam, rp, wq, total, map);
    RTP_CUDA(cudaGetLastError());
    ++*launches;
    { int rc = debug_sync(ds, st, "wave_generate_kernel", 0); if (rc != RTP_OK) return rc; }
    // a launch of at most tail_threshold paths (a 32x32 tile of main.rs:32, say) runs as generate + ONE tail-mode launch.
    // Offering every later queue of a big launch to the tail kernel was measured on C1 to be no faster than trace/shade
    // pairs, and so was handing the sparse late bounces to one tail launch chosen from the previous launch's queue sizes
    // (19 -> 12 launches per C1 frame, same 2.05 ms): a late bounce costs the latency of ONE ray segment (~30 us of
    // dependent instructions, tools/small_batches.py), not a launch. Tail mode maps paths to pixels densely and records no
    // first vertex: rtp_render only.
    if (std::is_same<Map, DenseTile>::value && !Aov::kOn && ds->sw.tail_threshold && total <= ds->sw.tail_threshold) {
        if (want_stats) next_mark(ds, st);  // even marks open a traversal span, odd marks close it
        const TailArgs ta{wq, rp, ds->scratch.ptr};
        if (int rc = launch_trace(ds, wq.rays[0], total, nullptr, OUT_TAIL, count, ds->counters, st, wq.count, &ta)) return rc;
        ++*launches;
        if (want_stats) next_mark(ds, st);
        return RTP_OK;
    }
    const unsigned shade_grid = static_cast<unsigned>(std::min<size_t>(static_cast<size_t>(ds->shade_blocks), (total + 255) / 256));
    for (uint32_t b = 0; b < rp.max_bounce; ++b) {
        if (want_stats) next_mark(ds, st);
        int rc = launch_trace(ds, wq.rays[b & 1], total, wq.hits, OUT_WAVE, count, ds->counters, st, wq.count + b);
        if (rc != RTP_OK) return rc;
        if (want_stats) next_mark(ds, st);
        if ((rc = debug_sync(ds, st, "trace kernel <OUT_WAVE>", b)) != RTP_OK) return rc;
        wave_shade_kernel<<<shade_grid, 256, 0, st>>>(ds->view, rp, wq, b, ds->scratch.ptr, map, aov);
        RTP_CUDA(cudaGetLastError());
        if ((rc = debug_sync(ds, st, "wave_shade_kernel", b)) != RTP_OK) return rc;
        *launches += ds->last_trace_launches + 1;
    }
    return RTP_OK;
}

// The AOV buffers of an rtp_render_aov call (device pointers, either may be null)
struct AovFrame {
    double* albedo;
    double* normal;
};

// aov != nullptr: an rtp_render_aov call. Its launches record every path's first vertex and never take tail mode; the records are
// folded into ds->aov_acc beside the colour and written to aov's buffers with the colour's divisor.
static int render_enqueue(DeviceScene* ds, const rtp_camera* camera, const rtp_render_params* p, double* d_rgb, double* d_fg, bool want_stats,
                          cudaStream_t st, uchar4* d_rgba8 = nullptr, const AovFrame* aov = nullptr) {
    DRender rp;
    if (int rc = render_begin(ds, p, true, want_stats, st, &rp)) return rc;
    const size_t npix = static_cast<size_t>(rp.tile_w) * rp.tile_h;
    const uint32_t ns_total = p->sample_end - p->sample_begin;
    size_t launches = 0;
    auto enqueue = [&]() -> int {
        if (npix == 0) return RTP_OK;  // no row of the rectangle falls to this call
        const uint32_t per_launch = static_cast<uint32_t>(std::max<size_t>(1, std::min<size_t>(ns_total ? ns_total : 1, path_budget(ds, p->max_bounce, aov != nullptr) / npix)));
        if (ns_total) {
            int rc = reserve_paths(ds, npix * per_launch, p->max_bounce, aov != nullptr);
            if (rc != RTP_OK) return rc;
        }
        if (int rc = ds->acc.reserve(npix)) return rc;
        if (aov) {
            if (int rc = ds->aov_acc.reserve(npix * 3)) return rc;
        }
        const bool count = (p->flags & RTP_RENDER_COUNTERS) != 0;
        const DCamera cam = make_camera(camera);

        bool first = true;
        if (ns_total == 0) RTP_CUDA(cudaMemsetAsync(ds->acc.ptr, 0, npix * sizeof(double4), st));
        if (ns_total == 0 && aov) RTP_CUDA(cudaMemsetAsync(ds->aov_acc.ptr, 0, npix * 3 * sizeof(double2), st));
        for (uint32_t s0 = 0; s0 < ns_total; s0 += per_launch) {
            rp.sample_begin = p->sample_begin + s0;
            rp.n_samples = std::min(per_launch, ns_total - s0);
            int rc = aov ? launch_paths(ds, cam, rp, DenseTile{}, AovRecords{ds->aov_rec.ptr}, npix * rp.n_samples, count, want_stats, st, &launches)
                         : launch_paths(ds, cam, rp, DenseTile{}, NoAov{}, npix * rp.n_samples, count, want_stats, st, &launches);
            if (rc != RTP_OK) return rc;
            resolve_kernel<<<static_cast<unsigned>((npix + 255) / 256), 256, 0, st>>>(ds->scratch.ptr, ds->acc.ptr, npix, rp.n_samples, first ? 1 : 0);
            RTP_CUDA(cudaGetLastError());
            ++launches;
            if (aov) {
                aov_resolve_kernel<<<static_cast<unsigned>((npix + 255) / 256), 256, 0, st>>>(ds->aov_rec.ptr, ds->aov_acc.ptr, npix, rp.n_samples, first ? 1 : 0);
                RTP_CUDA(cudaGetLastError());
                ++launches;
            }
            first = false;
        }
        const double divisor = (p->flags & RTP_RENDER_RAW_SUMS) ? 0.0 : static_cast<double>(p->num_samples);
        if (d_rgba8) {
            RTP_CUDA(cudaMemsetAsync(ds->n_fixes.ptr, 0, sizeof(unsigned int), st));
            srgb8_kernel<<<static_cast<unsigned>((npix + 255) / 256), 256, 0, st>>>(ds->acc.ptr, rp, divisor, (p->flags & RTP_RENDER_TRANSPARENT) ? 1 : 0, d_rgba8,
                                                                                    ds->fixes.ptr, ds->n_fixes.ptr, kSrgbFixCap);
        } else {
            write_frame_kernel<<<static_cast<unsigned>((npix + 255) / 256), 256, 0, st>>>(ds->acc.ptr, rp, divisor, d_rgb, d_fg);
        }
        RTP_CUDA(cudaGetLastError());
        ++launches;
        if (aov) {
            aov_write_kernel<<<static_cast<unsigned>((npix + 255) / 256), 256, 0, st>>>(ds->aov_acc.ptr, rp, divisor, aov->albedo, aov->normal);
            RTP_CUDA(cudaGetLastError());
            ++launches;
        }
        return RTP_OK;
    };
    const int rc = enqueue();
    const int rc_end = render_end(ds, st, want_stats, launches, static_cast<uint64_t>(npix) * ns_total);
    return rc != RTP_OK ? rc : rc_end;
}

// waits for the frame enqueued last on this device and fills `stats` (all fields)
static int render_finish(DeviceScene* ds, rtp_stats* stats) {
    RTP_CUDA(cudaEventSynchronize(ds->ev_end));
    if (int rc = read_stats(ds, stats)) return rc;
    double trace_ms = 0.0;
    for (size_t k = 0; k + 1 < ds->ev_used; k += 2) {
        float span = 0.f;
        if (cudaEventElapsedTime(&span, ds->ev_pool[k], ds->ev_pool[k + 1]) == cudaSuccess) trace_ms += span;
    }
    stats->paths = ds->pending_paths; stats->kernel_launches = ds->pending_launches;
    stats->trace_ms = trace_ms; stats->shade_ms = std::max(0.0, stats->device_ms - trace_ms);
    return RTP_OK;
}

static int render_device(rtp_scene* scene, const rtp_camera* camera, const rtp_render_params* p, double* d_rgb, double* d_fg, rtp_stats* stats,
                         cudaStream_t st, uchar4* d_rgba8 = nullptr, const AovFrame* aov = nullptr) {
    DeviceScene* ds = scene->dev;
    int rc = render_enqueue(ds, camera, p, d_rgb, d_fg, stats != nullptr, st, d_rgba8, aov);
    if (rc != RTP_OK) return rc;
    return stats ? render_finish(ds, stats) : RTP_OK;
}

// ---------------------------------------------------------------------------------------------
// rtp_render_adaptive (DESIGN.md §6b): rounds of samples over the pixels that are still live. Round 1 traces samples
// [0, min_samples) of every pixel, each later round the next min(batch, max_samples - n) samples of the live pixels. A round is
// split into launches by the path budget like rtp_render's sample range, each launch followed by adaptive_resolve_kernel; the last
// one decides the keep flags, a stable select builds the next live list and its length is read back. Tail mode is not used: it
// maps paths to pixels densely.
// ---------------------------------------------------------------------------------------------

static int check_adaptive(const rtp_render_params* p, const rtp_adaptive_params* a) {
    if (a->min_samples == 0 || a->min_samples > a->max_samples || a->batch == 0)
        return set_error(RTP_ERR_INVALID, "adaptive: need 0 < min_samples <= max_samples and batch > 0");
    if (!(a->abs_tol >= 0.0) || !(a->rel_tol >= 0.0) || std::isinf(a->abs_tol) || std::isinf(a->rel_tol))
        return set_error(RTP_ERR_INVALID, "adaptive: abs_tol and rel_tol must be finite and >= 0");
    if (p->num_samples || p->sample_begin || p->sample_end)
        return set_error(RTP_ERR_INVALID, "adaptive: the call owns the sample range; num_samples, sample_begin and sample_end must be 0");
    if (p->flags & ~(RTP_RENDER_RAW_SUMS | RTP_RENDER_COUNTERS))
        return set_error(RTP_ERR_INVALID, "adaptive: flags other than RTP_RENDER_RAW_SUMS | RTP_RENDER_COUNTERS");
    return RTP_OK;
}

// one device's share of an adaptive frame
struct AdaptiveDev {
    DeviceScene* ds = nullptr;
    cudaStream_t st = nullptr;
    const rtp_render_params* p = nullptr;  // this device's rows
    double* d_rgb = nullptr; double* d_fg = nullptr; uint32_t* d_samples = nullptr;
    DRender rp{};
    size_t npix = 0;
    uint32_t n_live = 0;    // length of live list `cur`
    int cur = 0;
    size_t launches = 0;
    uint64_t paths = 0;
};

// sizes the adaptive buffers for d's pixels and queues their initialisation: every pixel live, no sample yet
static int adaptive_init(AdaptiveDev& d) {
    DeviceScene* ds = d.ds;
    d.npix = static_cast<size_t>(d.rp.tile_w) * d.rp.tile_h;
    if (d.npix == 0) return RTP_OK;  // no row of the rectangle falls to this device
    if (d.npix > static_cast<size_t>(std::numeric_limits<int>::max()))  // cub::DeviceSelect counts items in int
        return set_error(RTP_ERR_UNSUPPORTED, "adaptive: more than 2^31 - 1 pixels on one device");
    int rc = ds->acc.reserve(d.npix);
    if (rc == RTP_OK) rc = ds->moments.reserve(d.npix);
    if (rc == RTP_OK) rc = ds->counts.reserve(d.npix);
    if (rc == RTP_OK) rc = ds->keep.reserve(d.npix);
    if (rc == RTP_OK) rc = ds->live[0].reserve(d.npix);
    if (rc == RTP_OK) rc = ds->live[1].reserve(d.npix);
    if (rc == RTP_OK) rc = ds->n_live.reserve(1);
    if (rc != RTP_OK) return rc;
    size_t tmp = 0;
    RTP_CUDA(cub::DeviceSelect::Flagged(nullptr, tmp, static_cast<const uint32_t*>(ds->live[0].ptr), ds->keep.ptr, ds->live[1].ptr, ds->n_live.ptr, static_cast<int>(d.npix), d.st));
    if ((rc = ds->select_tmp.reserve(tmp)) != RTP_OK) return rc;
    if (!ds->n_live_host) RTP_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&ds->n_live_host), sizeof(uint32_t), cudaHostAllocPortable));
    adaptive_init_kernel<<<static_cast<unsigned>((d.npix + 255) / 256), 256, 0, d.st>>>(ds->acc.ptr, ds->moments.ptr, ds->counts.ptr, ds->live[0].ptr, d.npix);
    RTP_CUDA(cudaGetLastError());
    ++d.launches;
    d.n_live = static_cast<uint32_t>(d.npix);
    d.cur = 0;
    return RTP_OK;
}

// queues samples [s0, s0 + B) of every live pixel, the stop rule and the selection of the next live list; its length is copied
// to ds->n_live_host
static int adaptive_round(AdaptiveDev& d, const DCamera& cam, uint32_t s0, uint32_t B, const StopRule& rule, bool count, bool want_stats) {
    DeviceScene* ds = d.ds;
    const uint32_t per_launch = static_cast<uint32_t>(std::max<size_t>(1, std::min<size_t>(B, path_budget(ds, d.rp.max_bounce) / d.n_live)));
    if (int rc = reserve_paths(ds, static_cast<size_t>(d.n_live) * per_launch, d.rp.max_bounce)) return rc;
    const LiveList map{ds->live[d.cur].ptr, d.n_live};
    const unsigned grid = (d.n_live + 255u) / 256u;
    for (uint32_t l0 = 0; l0 < B; l0 += per_launch) {
        d.rp.sample_begin = s0 + l0;
        d.rp.n_samples = std::min(per_launch, B - l0);
        int rc = launch_paths(ds, cam, d.rp, map, NoAov{}, static_cast<size_t>(d.n_live) * d.rp.n_samples, count, want_stats, d.st, &d.launches);
        if (rc != RTP_OK) return rc;
        adaptive_resolve_kernel<<<grid, 256, 0, d.st>>>(ds->scratch.ptr, map.live, d.n_live, d.rp.n_samples, ds->acc.ptr, ds->moments.ptr, ds->counts.ptr, ds->keep.ptr,
                                                        l0 + per_launch >= B ? 1 : 0, rule);
        RTP_CUDA(cudaGetLastError());
        ++d.launches;
    }
    d.paths += static_cast<uint64_t>(d.n_live) * B;
    size_t tmp = ds->select_tmp.n;
    RTP_CUDA(cub::DeviceSelect::Flagged(ds->select_tmp.ptr, tmp, map.live, ds->keep.ptr, ds->live[d.cur ^ 1].ptr, ds->n_live.ptr, static_cast<int>(d.n_live), d.st));
    d.launches += 2;  // the selection's scan-state initialisation and the select kernel
    RTP_CUDA(cudaMemcpyAsync(ds->n_live_host, ds->n_live.ptr, sizeof(uint32_t), cudaMemcpyDeviceToHost, d.st));
    d.cur ^= 1;
    return RTP_OK;
}

// Renders every device's share round by round: a round is queued on each device that still has live pixels, then every live count
// is read back. On return (also after an error) every device's work is queued and its output written or abandoned; the caller
// synchronises the streams.
static int render_adaptive(std::vector<AdaptiveDev>& devs, const rtp_camera* camera, const rtp_adaptive_params* a, bool want_stats) {
    const DCamera cam = make_camera(camera);
    const StopRule rule{a->abs_tol, a->rel_tol, a->max_samples, 0u};
    const bool count = (devs[0].p->flags & RTP_RENDER_COUNTERS) != 0;
    int rc = RTP_OK;
    size_t begun = 0;  // devs[0, begun) hold their scene's render scratch
    for (AdaptiveDev& d : devs) {
        if (cudaSetDevice(d.ds->device) != cudaSuccess) { rc = set_error(RTP_ERR_CUDA, "cudaSetDevice"); break; }
        if ((rc = render_begin(d.ds, d.p, false, want_stats, d.st, &d.rp)) != RTP_OK) break;
        ++begun;
        if ((rc = adaptive_init(d)) != RTP_OK) break;
    }
    uint32_t n = 0, B = a->min_samples;
    while (rc == RTP_OK) {
        bool queued = false;
        for (AdaptiveDev& d : devs) {
            if (rc != RTP_OK || d.n_live == 0) continue;
            cudaSetDevice(d.ds->device);
            rc = adaptive_round(d, cam, n, B, rule, count, want_stats);
            queued = true;
        }
        if (!queued) break;
        for (AdaptiveDev& d : devs) {
            if (d.n_live == 0) continue;
            cudaSetDevice(d.ds->device);
            const cudaError_t e = cudaStreamSynchronize(d.st);
            if (e != cudaSuccess && rc == RTP_OK) rc = set_error(RTP_ERR_CUDA, std::string("adaptive round: ") + cudaGetErrorString(e));
            d.n_live = rc == RTP_OK ? *d.ds->n_live_host : 0u;
        }
        n += B;
        if (n >= a->max_samples) break;  // the stop rule has stopped every pixel
        B = std::min(a->batch, a->max_samples - n);
    }
    const int raw = (devs[0].p->flags & RTP_RENDER_RAW_SUMS) ? 1 : 0;
    for (size_t k = 0; k < begun; ++k) {
        AdaptiveDev& d = devs[k];
        DeviceScene* ds = d.ds;
        cudaSetDevice(ds->device);
        if (rc == RTP_OK && d.npix) {
            adaptive_write_kernel<<<static_cast<unsigned>((d.npix + 255) / 256), 256, 0, d.st>>>(ds->acc.ptr, ds->counts.ptr, d.rp, raw, d.d_rgb, d.d_fg, d.d_samples);
            if (cudaGetLastError() != cudaSuccess) rc = set_error(RTP_ERR_CUDA, "adaptive_write_kernel launch");
            ++d.launches;
        }
        const int rc_end = render_end(ds, d.st, want_stats, d.launches, d.paths);
        if (rc == RTP_OK) rc = rc_end;
    }
    return rc;
}

// ---------------------------------------------------------------------------------------------
// The host-buffer render calls (rtp_render, rtp_render_srgb8, rtp_render_aov, rtp_render_adaptive) on one or several devices. The
// rows of the tile rectangle are dealt out round-robin to the devices taking part (params->device_mask); every device renders ALL
// samples of its rows into a frame-sized staging buffer, and only its rows travel back into the caller's frame: no exchange between
// devices, and since a pixel's value depends only on (seed, pixel, sample) the frame is bit-identical to a one-device render. All
// devices are driven from the calling thread: nothing is synchronised until every device's work is queued.
// ---------------------------------------------------------------------------------------------

// one device's share of a host-buffer render call
struct FrameDev {
    DeviceScene* ds;
    rtp_render_params p;  // the call's parameters with this device's rows
    std::unique_lock<std::mutex> lock;
};

// selects and locks the devices of params->device_mask (0: every device of the scene) and deals the rows out to them
static int deal_rows(rtp_scene* scene, const rtp_render_params* params, std::vector<FrameDev>* devs) {
    for (DeviceScene* ds : scene->devs)
        if (params->device_mask == 0 || ((params->device_mask >> ds->device) & 1u)) devs->push_back({ds, *params, std::unique_lock<std::mutex>(ds->lock)});
    if (devs->empty()) return set_error(RTP_ERR_INVALID, "device_mask names no device of this scene");
    const uint32_t N = static_cast<uint32_t>(devs->size());
    const uint32_t rs0 = params->row_stride ? params->row_stride : 1u;
    for (uint32_t k = 0; k < N; ++k) {
        rtp_render_params& p = (*devs)[k].p;
        p.row_offset = params->row_offset + k * rs0;  // rows ro0 + m * rs0 of the caller's split; device k takes m = k, k + N, ...
        p.row_stride = rs0 * N;
    }
    return RTP_OK;
}

// one plane of a frame: the caller's buffer (nullptr: not asked for), the device's frame-sized staging buffer, bytes per pixel
struct Plane {
    void* host;
    const void* dev;
    size_t px_bytes;
};

// queues on `st` the copy of the rows `p` covers (main.rs:86-87 writes per tile) from the device's planes into the caller's
static int copy_rows(const rtp_render_params& p, cudaStream_t st, std::initializer_list<Plane> planes) {
    DRender rp;
    if (int rc = render_rect(&p, false, &rp)) return rc;
    if (rp.tile_h == 0) return RTP_OK;  // no row of the rectangle fell to this device
    const size_t first = rp.tile_x + static_cast<size_t>(rp.tile_y + rp.row_offset) * rp.width;
    const size_t row_px = static_cast<size_t>(rp.width) * rp.row_stride;
    for (const Plane& pl : planes) {
        if (!pl.host) continue;
        const size_t b = pl.px_bytes;
        const cudaError_t e = cudaMemcpy2DAsync(static_cast<char*>(pl.host) + first * b, row_px * b, static_cast<const char*>(pl.dev) + first * b, row_px * b,
                                                rp.tile_w * b, rp.tile_h, cudaMemcpyDeviceToHost, st);
        if (e != cudaSuccess) return set_error(RTP_ERR_CUDA, std::string("frame copy: ") + cudaGetErrorString(e));
    }
    return RTP_OK;
}

// rtp_render_srgb8 on a finished device: redoes its borderline pixels with the host libm (utility.rs:213 powf as the reference's
// target evaluates it)
static int srgb_fixup(const DeviceScene* ds, uint8_t* rgba_out) {
    const unsigned int n_fix = ds->n_fix_host;
    if (n_fix > kSrgbFixCap) return set_error(RTP_ERR_UNSUPPORTED, "more than 65536 pixels need the host libm fix-up; use rtp_render + rtp_frame_to_srgb8");
    if (n_fix == 0) return RTP_OK;
    std::vector<SrgbFix> fixes(n_fix);
    if (cudaMemcpy(fixes.data(), ds->fixes.ptr, n_fix * sizeof(SrgbFix), cudaMemcpyDeviceToHost) != cudaSuccess) return set_error(RTP_ERR_CUDA, "fix-up list copy");
    for (const SrgbFix& f : fixes) {
        uint8_t px[4];
        rtp_frame_to_srgb8(f.rgb, 1, 1, px);
        std::memcpy(rgba_out + 4 * static_cast<size_t>(f.pixel), px, 3);
    }
    return RTP_OK;
}

// Waits for every device of the call, also after an error on another one (nothing may stay in flight on a scene's scratch), then
// applies the sRGB fix-up (rgba_out != nullptr) and sums the devices' stats. Leaves the scene's first device current.
static int finish_frame(rtp_scene* scene, std::vector<FrameDev>& devs, int rc, rtp_stats* stats, uint8_t* rgba_out) {
    rtp_stats total;
    std::memset(&total, 0, sizeof total);
    for (FrameDev& d : devs) {
        DeviceScene* ds = d.ds;
        cudaSetDevice(ds->device);
        const cudaError_t e = cudaStreamSynchronize(ds->streams[0]);
        if (e != cudaSuccess && rc == RTP_OK) rc = set_error(RTP_ERR_CUDA, std::string("render: ") + cudaGetErrorString(e));
        if (rc == RTP_OK && rgba_out && ds->pending_launches) rc = srgb_fixup(ds, rgba_out);
        if (rc != RTP_OK || !stats) continue;
        rtp_stats one;
        if ((rc = render_finish(ds, &one)) == RTP_OK) add_stats(&total, one);
    }
    cudaSetDevice(scene->dev->device);
    if (stats && rc == RTP_OK) *stats = total;
    return rc;
}

}  // namespace rtp

// =============================================================================================
// C ABI — device entry points
// =============================================================================================

using namespace rtp;

extern "C" {

int rtp_device_count(int* count) {
    if (!count) return set_error(RTP_ERR_INVALID, "null argument");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { *count = 0; return set_error(RTP_ERR_CUDA, std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e)); }
    *count = n;
    return RTP_OK;
}

int rtp_init(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return set_error(RTP_ERR_CUDA, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                                           " (this library has no CPU fallback)");
    if (device < 0 || device >= n) return set_error(RTP_ERR_INVALID, "device index out of range");
    cudaDeviceProp prop;
    RTP_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return set_error(RTP_ERR_CUDA, std::string("device ") + prop.name + " is not compute capability 10.x; kernels are built for sm_100a only");
    RTP_CUDA(cudaSetDevice(device));
    RTP_CUDA(cudaFree(nullptr));
    g_device = device;
    return RTP_OK;
}

int rtp_scene_digest(const rtp_scene* scene, uint64_t digest_out[4]) {
    if (!scene || !digest_out || !scene->dev) return set_error(RTP_ERR_INVALID, "null argument");
    const DeviceScene* ds = scene->dev;
    RTP_CUDA(cudaSetDevice(ds->device));
    const size_t n_nodes = ds->view.n_nodes, n_prims = ds->view.n_prims, n_wide = ds->n_wide;
    auto fnv = [](uint64_t h, const void* p, size_t bytes) {
        const unsigned char* b = static_cast<const unsigned char*>(p);
        for (size_t i = 0; i < bytes; ++i) { h ^= b[i]; h *= 0x100000001B3ull; }
        return h;
    };
    try {
        std::vector<DNode> nodes(n_nodes);
        if (n_nodes) RTP_CUDA(cudaMemcpy(nodes.data(), ds->nodes, n_nodes * sizeof(DNode), cudaMemcpyDeviceToHost));
        uint64_t h0 = 0xCBF29CE484222325ull;
        // the sign of a zero coordinate is not part of the tree: IEEE minNum / maxNum may return either of -0.0 and +0.0 (libm's
        // fmin and the device's differ), and no slab test can tell them apart; x + 0.0 maps both to +0.0. _pad is build-private.
        for (const DNode& nd : nodes) {
            double box[6];
            for (int k = 0; k < 3; ++k) { box[k] = nd.bmin[k] + 0.0; box[3 + k] = nd.bmax[k] + 0.0; }
            h0 = fnv(h0, box, 48); h0 = fnv(h0, &nd.skip, 12);
        }
        std::vector<DNode>().swap(nodes);
        uint64_t h1 = 0xCBF29CE484222325ull;
        {
            std::vector<DPrim> prims(n_prims);
            if (n_prims) RTP_CUDA(cudaMemcpy(prims.data(), ds->prims, n_prims * sizeof(DPrim), cudaMemcpyDeviceToHost));
            h1 = fnv(h1, prims.data(), n_prims * sizeof(DPrim));
        }
        {
            std::vector<DAttr> attrs(n_prims);
            if (n_prims) RTP_CUDA(cudaMemcpy(attrs.data(), ds->attrs, n_prims * sizeof(DAttr), cudaMemcpyDeviceToHost));
            h1 = fnv(h1, attrs.data(), n_prims * sizeof(DAttr));
        }
        // a 4-wide tree hashed from its root down: a node's hash folds its planes and, per child, the leaf word or the child's hash
        // (post-order from node 0), so that the numbering of the nodes does not matter. Returns 0 and sets *bad on a dangling child.
        auto tree_hash = [&](const DWide* d_wide, size_t n, uint32_t* levels, bool* bad) -> uint64_t {
            std::vector<DWide> wide(n);
            if (n && cudaMemcpy(wide.data(), d_wide, n * sizeof(DWide), cudaMemcpyDeviceToHost) != cudaSuccess) { *bad = true; return 0; }
            std::vector<uint64_t> hash(n, 0);
            std::vector<uint8_t> done(n, 0);
            std::vector<uint32_t> stack, depth_of(n, 0);
            *levels = 0;
            if (n) { stack.push_back(0); depth_of[0] = 1; }
            while (!stack.empty()) {
                const uint32_t i = stack.back();
                bool ready = true;
                for (int k = 0; k < 4; ++k) {
                    const uint32_t c = wide[i].child[k];
                    if (!(c & kWideLeaf) && !done[c]) { if (c >= n) { *bad = true; return 0; } depth_of[c] = depth_of[i] + 1; stack.push_back(c); ready = false; }
                }
                if (!ready) continue;
                stack.pop_back();
                float planes[24];
                for (int k = 0; k < 24; ++k) planes[k] = (&wide[i].plane[0][0][0])[k] + 0.0f;
                uint64_t h = fnv(0xCBF29CE484222325ull, planes, sizeof planes);
                for (int k = 0; k < 4; ++k) {
                    const uint32_t c = wide[i].child[k];
                    const uint64_t v = (c & kWideLeaf) ? static_cast<uint64_t>(c) : hash[c];
                    h = fnv(h, &v, 8);
                }
                hash[i] = h; done[i] = 1;
                *levels = std::max(*levels, depth_of[i]);
            }
            return n ? hash[0] : 0;
        };
        uint32_t levels = 0, free_levels = 0;
        bool bad = false;
        uint64_t h2 = tree_hash(ds->wide, n_wide, &levels, &bad);
        if (n_wide) {  // the culled-set box belongs to the culling tree
            float cull[6];
            for (int k = 0; k < 6; ++k) cull[k] = ds->view.cull[k] + 0.0f;
            h2 = fnv(h2, cull, sizeof cull);
        }
        if (ds->free_wide) {  // and so does the order-free tree of the any-order lanes
            const uint64_t hf = tree_hash(ds->free_wide, ds->n_free_wide, &free_levels, &bad);
            h2 = fnv(h2, &hf, 8);
        }
        if (bad) return set_error(RTP_ERR_INVALID, "4-wide tree: child index out of range or unreadable");
        digest_out[0] = h0; digest_out[1] = h1; digest_out[2] = h2; digest_out[3] = static_cast<uint64_t>(n_wide) | (static_cast<uint64_t>(levels) << 32);
    } catch (const std::exception& e) {
        return set_error(RTP_ERR_NOMEM, e.what());
    }
    return RTP_OK;
}

int rtp_scene_any_tables(const rtp_scene* scene, rtp_any_tables* out) {
    if (!scene || !out) return set_error(RTP_ERR_INVALID, "null argument");
    const FlatScene& f = scene->flat;
    std::memset(out, 0, sizeof *out);
    out->n_big = f.n_big;
    for (int k = 0; k < 8; ++k) out->big[k] = f.big[k];
    out->any_spheres = f.any_spheres ? 1u : 0u;
    out->any_E = f.any_E; out->any_A = f.any_A; out->any_C = f.any_C; out->any_R = f.any_R;
    out->scene_mag = f.scene_mag;
    for (int k = 0; k < 6; ++k) out->cull[k] = f.cull[k];
    return RTP_OK;
}

int rtp_probe_fp64(double* gops_out) {
    if (!gops_out) return set_error(RTP_ERR_INVALID, "null argument");
    int rc = require_device();
    if (rc != RTP_OK) return rc;
    cudaDeviceProp prop;
    RTP_CUDA(cudaGetDeviceProperties(&prop, g_device));
    double* sink = nullptr;
    RTP_CUDA(cudaMalloc(reinterpret_cast<void**>(&sink), sizeof(double) * 4096));
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    cudaError_t e = cudaEventCreate(&e0);
    if (e == cudaSuccess) e = cudaEventCreate(&e1);
    const int blocks = prop.multiProcessorCount * 8, iters = 16384;
    double best = 0.0;
    for (int rep = 0; rep < 4 && e == cudaSuccess; ++rep) {  // first repetition warms up
        cudaEventRecord(e0);
        fp64_probe_kernel<<<blocks, 256>>>(sink, 0.999999, 1e-6, iters);
        cudaEventRecord(e1);
        e = cudaEventSynchronize(e1);
        float ms = 0.f;
        if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
        if (e == cudaSuccess && rep > 0 && ms > 0.f) best = std::max(best, 2.0 * 8.0 * iters * 256.0 * blocks / (ms * 1e-3) / 1e9);
    }
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    cudaFree(sink);
    if (e != cudaSuccess) return set_error(RTP_ERR_CUDA, std::string("fp64 probe: ") + cudaGetErrorString(e));
    *gops_out = best;
    return RTP_OK;
}

int rtp_host_alloc(size_t bytes, void** out) {
    if (!out) return set_error(RTP_ERR_INVALID, "null argument");
    int rc = require_device();
    if (rc != RTP_OK) return rc;
    RTP_CUDA(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
    return RTP_OK;
}

void rtp_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

// device_mask == 0: the device bound by rtp_init (or device 0)
static int scene_create_impl(const rtp_scene_desc* desc, uint32_t device_mask, rtp_scene** out) {
    if (!out) return set_error(RTP_ERR_INVALID, "null argument");
    *out = nullptr;
    try {
        rtp_scene* s = new rtp_scene();
        auto bail = [&](int code) { for (DeviceScene* ds : s->devs) { cudaSetDevice(ds->device); device_scene_free(ds); } device_free_arrays(&s->flat.dev); delete s; return code; };
        int rc = RTP_OK;
        if (device_mask) {
            for (int d = 0; d < 32 && rc == RTP_OK; ++d)
                if ((device_mask >> d) & 1u) rc = check_device(d);
            if (rc != RTP_OK) return bail(rc);
            int first = 0;
            while (!((device_mask >> first) & 1u)) ++first;
            if (g_device < 0) g_device = first;
            cudaSetDevice(first);  // the device part of the build (reference leaf order of big scenes) runs on the first device
        }
        const Switches sw = read_switches();
        rc = flatten_scene(desc, sw, &s->flat, /*device_build=*/true);  // validates before it touches the device
        if (rc != RTP_OK) return bail(rc);
        if (!device_mask) {
            if ((rc = require_device()) != RTP_OK) return bail(rc);
            device_mask = 1u << g_device;
        }
        for (int d = 0; d < 32 && rc == RTP_OK; ++d)
            if ((device_mask >> d) & 1u) {
                DeviceScene* ds = nullptr;
                rc = device_scene_upload(s->flat, sw, d, &ds);
                if (rc == RTP_OK) s->devs.push_back(ds);
            }
        if (rc != RTP_OK) return bail(rc);
        s->dev = s->devs[0];
        cudaSetDevice(s->dev->device);
        s->n_leaves = static_cast<uint32_t>(s->flat.prim_count());
        device_free_arrays(&s->flat.dev);  // every replica holds its own copy now
        s->n_nodes = s->flat.root_kind == RTP_ROOT_BVH ? s->flat.n_reference_nodes : 0u;
        // the host copies of the big arrays are no longer needed
        std::vector<DNode>().swap(s->flat.nodes);
        std::vector<DWide>().swap(s->flat.wide);
        std::vector<double>().swap(s->flat.wide_boxes);
        std::vector<DWide>().swap(s->flat.free_wide);
        std::vector<double>().swap(s->flat.free_boxes);
        std::vector<DPrim>().swap(s->flat.prims);
        std::vector<DAttr>().swap(s->flat.attrs);
        std::vector<std::vector<uint8_t>>().swap(s->flat.images);
        *out = s;
        return RTP_OK;
    } catch (const std::exception& e) {
        return set_error(RTP_ERR_NOMEM, e.what());
    }
}

int rtp_scene_create_multi(const rtp_scene_desc* desc, uint32_t device_mask, rtp_scene** out) {
    if (device_mask == 0) { if (out) *out = nullptr; return set_error(RTP_ERR_INVALID, "empty device mask"); }
    return scene_create_impl(desc, device_mask, out);
}

int rtp_scene_create(const rtp_scene_desc* desc, rtp_scene** out) { return scene_create_impl(desc, 0u, out); }

int rtp_scene_devices(const rtp_scene* scene, uint32_t* device_mask_out) {
    if (!scene || !device_mask_out) return set_error(RTP_ERR_INVALID, "null argument");
    uint32_t m = 0;
    for (const DeviceScene* ds : scene->devs) m |= 1u << ds->device;
    *device_mask_out = m;
    return RTP_OK;
}

void rtp_scene_destroy(rtp_scene* scene) {
    if (!scene) return;
    const int primary = scene->dev ? scene->dev->device : -1;
    for (DeviceScene* ds : scene->devs) { cudaSetDevice(ds->device); device_scene_free(ds); }
    if (primary >= 0) cudaSetDevice(primary);
    delete scene;
}

int rtp_scene_get_info(const rtp_scene* scene, rtp_scene_info* info) {
    if (!scene || !info) return set_error(RTP_ERR_INVALID, "null argument");
    info->n_leaves = scene->n_leaves; info->n_nodes = scene->n_nodes;
    info->depth = scene->flat.depth; info->root_kind = scene->flat.root_kind;
    info->device_bytes = device_scene_bytes(scene->dev);
    info->culling_depth = scene->flat.root_kind == RTP_ROOT_BVH ? scene->flat.wide_depth : 0u;
    info->any_order = scene->dev ? static_cast<uint32_t>(scene->dev->any_order) : 0u;
    info->n_big = scene->flat.n_big; info->free_tree_depth = scene->flat.free_depth;
    return RTP_OK;
}

int rtp_bvh_build_order(const rtp_scene_desc* desc, uint32_t* leaf_ids_out, size_t cap, rtp_scene_info* info) {
    try {
        FlatScene flat;
        int rc = flatten_scene(desc, read_switches(), &flat);
        if (rc != RTP_OK) return rc;
        if (leaf_ids_out) {
            if (cap < flat.leaf_order.size()) return set_error(RTP_ERR_INVALID, "leaf_ids_out too small");
            std::copy(flat.leaf_order.begin(), flat.leaf_order.end(), leaf_ids_out);
        }
        if (info) {
            info->n_leaves = static_cast<uint32_t>(flat.prim_count());
            info->n_nodes = flat.root_kind == RTP_ROOT_BVH ? flat.n_reference_nodes : 0u;
            info->depth = flat.depth; info->root_kind = flat.root_kind; info->device_bytes = 0;
            info->culling_depth = flat.root_kind == RTP_ROOT_BVH ? flat.wide_depth : 0u;
            info->any_order = flat.any_ok ? 1u : 0u; info->n_big = flat.n_big; info->free_tree_depth = flat.free_depth;
        }
        return RTP_OK;
    } catch (const std::exception& e) {
        return set_error(RTP_ERR_NOMEM, e.what());
    }
}

int rtp_bvh_culled_set(const rtp_scene_desc* desc, float box_out[6], uint32_t* free_tree_leaves, uint32_t* free_tree_big_leaves) {
    if (!box_out || !free_tree_leaves || !free_tree_big_leaves) return set_error(RTP_ERR_INVALID, "null argument");
    try {
        FlatScene flat;
        int rc = flatten_scene(desc, read_switches(), &flat);
        if (rc != RTP_OK) return rc;
        std::copy(flat.cull, flat.cull + 6, box_out);
        uint32_t leaves = 0, big = 0;
        for (const DWide& w : flat.free_wide)
            for (int k = 0; k < 4; ++k) {
                const uint32_t c = w.child[k];
                if (c == kWideEmpty || !(c & kWideLeaf)) continue;
                ++leaves;
                for (uint32_t q = 0; q < flat.n_big; ++q) big += (flat.big[q] & kWideSlotMask) == (c & kWideSlotMask) ? 1u : 0u;
            }
        *free_tree_leaves = leaves; *free_tree_big_leaves = big;
        return RTP_OK;
    } catch (const std::exception& e) {
        return set_error(RTP_ERR_NOMEM, e.what());
    }
}

int rtp_scene_leaf_order(const rtp_scene* scene, uint32_t* out, size_t cap) {
    if (!scene || !out || cap < scene->flat.leaf_order.size()) return set_error(RTP_ERR_INVALID, "bad argument");
    std::copy(scene->flat.leaf_order.begin(), scene->flat.leaf_order.end(), out);
    return RTP_OK;
}

int rtp_trace_closest(rtp_scene* scene, const rtp_ray* rays, size_t n, rtp_hit* hits_out, rtp_stats* stats) {
    if (!scene || (n && (!rays || !hits_out))) return set_error(RTP_ERR_INVALID, "null argument");
    if (stats) std::memset(stats, 0, sizeof *stats);
    if (n == 0) return RTP_OK;
    return trace_host(scene, rays, n, hits_out, OUT_HIT, stats);
}

int rtp_trace_closest_full(rtp_scene* scene, const rtp_ray* rays, size_t n, rtp_hit_full* hits_out, rtp_stats* stats) {
    if (!scene || (n && (!rays || !hits_out))) return set_error(RTP_ERR_INVALID, "null argument");
    if (stats) std::memset(stats, 0, sizeof *stats);
    if (n == 0) return RTP_OK;
    return trace_host(scene, rays, n, hits_out, OUT_FULL, stats);
}

int rtp_trace_camera(rtp_scene* scene, const rtp_camera* camera, uint32_t width, uint32_t height, rtp_hit* hits_out, rtp_stats* stats) {
    if (!scene || !camera || !hits_out) return set_error(RTP_ERR_INVALID, "null argument");
    if (stats) std::memset(stats, 0, sizeof *stats);
    const size_t n = static_cast<size_t>(width) * height;
    if (n == 0) return RTP_OK;
    const DCamera cam = make_camera(camera);
    return trace_host(scene, nullptr, n, hits_out, OUT_HIT, stats, &cam, width, height);
}

int rtp_trace_closest_device(rtp_scene* scene, const rtp_ray* d_rays, size_t n, rtp_hit* d_hits_out, void* cuda_stream) {
    if (!scene || (n && (!d_rays || !d_hits_out))) return set_error(RTP_ERR_INVALID, "null argument");
    RTP_CUDA(cudaSetDevice(scene->dev->device));
    return launch_trace(scene->dev, d_rays, n, d_hits_out, OUT_HIT, false, nullptr, static_cast<cudaStream_t>(cuda_stream));
}

/* Counting variant used by tests and the roofline report: node visits / primitive tests for a device-resident batch. */
static int trace_device_counted(rtp_scene* scene, const rtp_ray* d_rays, size_t n, void* d_out, int out_mode, rtp_stats* stats) {
    DeviceScene* ds = scene->dev;
    std::lock_guard<std::mutex> guard(ds->lock);
    RTP_CUDA(cudaSetDevice(ds->device));
    cudaStream_t st = ds->streams[0];
    RTP_CUDA(cudaMemsetAsync(ds->counters, 0, sizeof(Counters), st));
    RTP_CUDA(cudaEventRecord(ds->ev_begin, st));
    int rc = launch_trace(ds, d_rays, n, d_out, out_mode, true, ds->counters, st);
    if (rc != RTP_OK) return rc;
    RTP_CUDA(cudaEventRecord(ds->ev_end, st));
    RTP_CUDA(cudaEventSynchronize(ds->ev_end));
    Counters c;
    if ((rc = read_stats(ds, stats, &c)) != RTP_OK) return rc;
    stats->kernel_launches = 1;
    if (ds->sw.lane_stats && c.rounds)
        std::fprintf(stderr, "[rtp lanes] %llu rounds (%.1f per ray): per round %.1f lanes can walk, %.1f hold two leaves, %.1f wait for a leaf test with nothing left to walk, %.1f hold no ray; "
                             "%llu leaf rounds at %.1f lanes\n", c.rounds, double(c.rounds) * 32.0 / double(c.rays ? c.rays : 1), double(c.lanes_walk) / c.rounds, double(c.lanes_full) / c.rounds,
                     double(c.lanes_leafwait) / c.rounds, double(c.lanes_empty) / c.rounds, c.leaf_rounds, c.leaf_rounds ? double(c.leaf_lanes) / c.leaf_rounds : 0.0);
    return RTP_OK;
}

int rtp_trace_closest_device_counted(rtp_scene* scene, const rtp_ray* d_rays, size_t n, rtp_hit* d_hits_out, rtp_stats* stats) {
    if (!scene || !stats || (n && (!d_rays || !d_hits_out))) return set_error(RTP_ERR_INVALID, "null argument");
    return trace_device_counted(scene, d_rays, n, d_hits_out, OUT_HIT, stats);
}

// Occlusion (DESIGN.md §2c): the in-order walk with T fixed at ray.t_max, stopped at the first accepted leaf; one byte per ray
int rtp_trace_occluded(rtp_scene* scene, const rtp_ray* rays, size_t n, uint8_t* occluded_out, rtp_stats* stats) {
    if (!scene || (n && (!rays || !occluded_out))) return set_error(RTP_ERR_INVALID, "null argument");
    if (stats) std::memset(stats, 0, sizeof *stats);
    if (n == 0) return RTP_OK;
    return trace_host(scene, rays, n, occluded_out, OUT_OCCLUDED, stats);
}

int rtp_trace_occluded_device(rtp_scene* scene, const rtp_ray* d_rays, size_t n, uint8_t* d_occluded_out, void* cuda_stream) {
    if (!scene || (n && (!d_rays || !d_occluded_out))) return set_error(RTP_ERR_INVALID, "null argument");
    if (n == 0) return RTP_OK;
    RTP_CUDA(cudaSetDevice(scene->dev->device));
    return launch_trace(scene->dev, d_rays, n, d_occluded_out, OUT_OCCLUDED, false, nullptr, static_cast<cudaStream_t>(cuda_stream));
}

int rtp_trace_occluded_device_counted(rtp_scene* scene, const rtp_ray* d_rays, size_t n, uint8_t* d_occluded_out, rtp_stats* stats) {
    if (!scene || !stats || (n && (!d_rays || !d_occluded_out))) return set_error(RTP_ERR_INVALID, "null argument");
    std::memset(stats, 0, sizeof *stats);
    if (n == 0) return RTP_OK;
    return trace_device_counted(scene, d_rays, n, d_occluded_out, OUT_OCCLUDED, stats);
}

int rtp_camera_rays_device(const rtp_camera* camera, uint32_t width, uint32_t height, rtp_ray* d_rays_out, void* cuda_stream) {
    if (!camera || !d_rays_out) return set_error(RTP_ERR_INVALID, "null argument");
    int rc = require_device();
    if (rc != RTP_OK) return rc;
    const size_t n = static_cast<size_t>(width) * height;
    if (n == 0) return RTP_OK;
    const DCamera cam = make_camera(camera);
    camera_rays_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(cam, width, height, d_rays_out, 0, n);
    RTP_CUDA(cudaGetLastError());
    return RTP_OK;
}

int rtp_camera_rays(const rtp_camera* camera, uint32_t width, uint32_t height, rtp_ray* rays_out) {
    if (!camera || !rays_out) return set_error(RTP_ERR_INVALID, "null argument");
    int rc = require_device();
    if (rc != RTP_OK) return rc;
    const size_t n = static_cast<size_t>(width) * height;
    if (n == 0) return RTP_OK;
    rtp_ray* d = nullptr;
    RTP_CUDA(cudaMalloc(reinterpret_cast<void**>(&d), n * sizeof(rtp_ray)));
    rc = rtp_camera_rays_device(camera, width, height, d, nullptr);
    cudaError_t e = rc == RTP_OK ? cudaMemcpy(rays_out, d, n * sizeof(rtp_ray), cudaMemcpyDeviceToHost) : cudaSuccess;
    cudaFree(d);
    if (rc != RTP_OK) return rc;
    if (e != cudaSuccess) return set_error(RTP_ERR_CUDA, std::string("camera rays copy: ") + cudaGetErrorString(e));
    return RTP_OK;
}

int rtp_render_device(rtp_scene* scene, const rtp_camera* camera, const rtp_render_params* params, double* d_rgb_out, double* d_foreground_out,
                      rtp_stats* stats, void* cuda_stream) {
    if (!scene || !camera || !params || !d_rgb_out) return set_error(RTP_ERR_INVALID, "null argument");
    DeviceScene* ds = scene->dev;
    std::lock_guard<std::mutex> guard(ds->lock);
    RTP_CUDA(cudaSetDevice(ds->device));
    return render_device(scene, camera, params, d_rgb_out, d_foreground_out, stats, static_cast<cudaStream_t>(cuda_stream));
}

// rtp_render / rtp_render_srgb8 / rtp_render_aov with host buffers, on the devices of params->device_mask (see deal_rows).
// aov != nullptr (host pointers, either may be null): an rtp_render_aov call, whose staging frame holds 6 more doubles per pixel.
static int render_host(rtp_scene* scene, const rtp_camera* camera, const rtp_render_params* params, double* rgb_out, double* foreground_out,
                       uint8_t* rgba_out, rtp_stats* stats, const AovFrame* aov = nullptr) {
    const size_t npx = static_cast<size_t>(params->width) * params->height;
    if (npx == 0) return set_error(RTP_ERR_INVALID, "bad frame parameters");
    std::vector<FrameDev> devs;
    if (int rc = deal_rows(scene, params, &devs)) return rc;
    int rc = RTP_OK;
    for (FrameDev& d : devs) {
        DeviceScene* ds = d.ds;
        cudaStream_t st = ds->streams[0];
        if (cudaSetDevice(ds->device) != cudaSuccess) { rc = set_error(RTP_ERR_CUDA, "cudaSetDevice"); break; }
        if (rgba_out) {
            rc = ds->frame8.reserve(npx);
            if (rc == RTP_OK) rc = ds->fixes.reserve(kSrgbFixCap);
            if (rc == RTP_OK) rc = ds->n_fixes.reserve(1);
            if (rc == RTP_OK) rc = render_enqueue(ds, camera, &d.p, nullptr, nullptr, stats != nullptr, st, ds->frame8.ptr);
            if (rc == RTP_OK) rc = copy_rows(d.p, st, {{rgba_out, ds->frame8.ptr, 4}});
            if (rc == RTP_OK && ds->pending_launches) {
                const cudaError_t e = cudaMemcpyAsync(&ds->n_fix_host, ds->n_fixes.ptr, sizeof(unsigned int), cudaMemcpyDeviceToHost, st);
                if (e != cudaSuccess) rc = set_error(RTP_ERR_CUDA, std::string("fix-up count copy: ") + cudaGetErrorString(e));
            }
        } else {
            if ((rc = ds->frame.reserve(npx * (aov ? 10 : 4))) != RTP_OK) break;  // rgb, foreground [, albedo, normal]
            double* f = ds->frame.ptr;
            const AovFrame d_aov = {aov && aov->albedo ? f + npx * 4 : nullptr, aov && aov->normal ? f + npx * 7 : nullptr};
            rc = render_enqueue(ds, camera, &d.p, f, foreground_out ? f + npx * 3 : nullptr, stats != nullptr, st, nullptr, aov ? &d_aov : nullptr);
            if (rc == RTP_OK)
                rc = copy_rows(d.p, st, {{rgb_out, f, 24}, {foreground_out, f + npx * 3, 8}, {d_aov.albedo ? aov->albedo : nullptr, d_aov.albedo, 24},
                                         {d_aov.normal ? aov->normal : nullptr, d_aov.normal, 24}});
        }
        if (rc != RTP_OK) break;
    }
    return finish_frame(scene, devs, rc, stats, rgba_out);
}

int rtp_render_srgb8(rtp_scene* scene, const rtp_camera* camera, const rtp_render_params* params, uint8_t* rgba_out, rtp_stats* stats) {
    if (!scene || !camera || !params || !rgba_out) return set_error(RTP_ERR_INVALID, "null argument");
    if (params->flags & RTP_RENDER_RAW_SUMS) return set_error(RTP_ERR_INVALID, "RTP_RENDER_RAW_SUMS has no 8-bit output");
    return render_host(scene, camera, params, nullptr, nullptr, rgba_out, stats);
}

int rtp_render(rtp_scene* scene, const rtp_camera* camera, const rtp_render_params* params, double* rgb_out, double* foreground_out,
               rtp_stats* stats) {
    if (!scene || !camera || !params || !rgb_out) return set_error(RTP_ERR_INVALID, "null argument");
    return render_host(scene, camera, params, rgb_out, foreground_out, nullptr, stats);
}

// rtp_render plus each pixel's mean first-vertex albedo and normal (DESIGN.md §6c)
static int check_aov(const rtp_scene* scene, const rtp_camera* camera, const rtp_render_params* params, const double* rgb_out) {
    if (!scene || !camera || !params || !rgb_out) return set_error(RTP_ERR_INVALID, "null argument");
    if (params->flags & ~(RTP_RENDER_RAW_SUMS | RTP_RENDER_COUNTERS))
        return set_error(RTP_ERR_INVALID, "aov: flags other than RTP_RENDER_RAW_SUMS | RTP_RENDER_COUNTERS");
    return RTP_OK;
}

int rtp_render_aov(rtp_scene* scene, const rtp_camera* camera, const rtp_render_params* params, double* rgb_out, double* foreground_out,
                   double* albedo_out, double* normal_out, rtp_stats* stats) {
    if (int rc = check_aov(scene, camera, params, rgb_out)) return rc;
    const AovFrame aov = {albedo_out, normal_out};
    return render_host(scene, camera, params, rgb_out, foreground_out, nullptr, stats, &aov);
}

int rtp_render_aov_device(rtp_scene* scene, const rtp_camera* camera, const rtp_render_params* params, double* d_rgb_out, double* d_foreground_out,
                          double* d_albedo_out, double* d_normal_out, rtp_stats* stats, void* cuda_stream) {
    if (int rc = check_aov(scene, camera, params, d_rgb_out)) return rc;
    DeviceScene* ds = scene->dev;
    std::lock_guard<std::mutex> guard(ds->lock);
    RTP_CUDA(cudaSetDevice(ds->device));
    const AovFrame aov = {d_albedo_out, d_normal_out};
    return render_device(scene, camera, params, d_rgb_out, d_foreground_out, stats, static_cast<cudaStream_t>(cuda_stream), nullptr, &aov);
}

// The rows of the tile rectangle are dealt out to the devices as in render_host; each device runs its own live list through the same
// rounds, and only its rows travel back.
int rtp_render_adaptive(rtp_scene* scene, const rtp_camera* camera, const rtp_render_params* params, const rtp_adaptive_params* adaptive,
                        double* rgb_out, double* foreground_out, uint32_t* samples_out, rtp_stats* stats) {
    if (!scene || !camera || !params || !adaptive || !rgb_out) return set_error(RTP_ERR_INVALID, "null argument");
    if (int rc = check_adaptive(params, adaptive)) return rc;
    const size_t npx = static_cast<size_t>(params->width) * params->height;
    if (npx == 0) return set_error(RTP_ERR_INVALID, "bad frame parameters");
    std::vector<FrameDev> frame;
    if (int rc = deal_rows(scene, params, &frame)) return rc;
    std::vector<AdaptiveDev> devs(frame.size());
    int rc = RTP_OK;
    for (size_t k = 0; k < frame.size() && rc == RTP_OK; ++k) {
        AdaptiveDev& d = devs[k];
        DeviceScene* ds = frame[k].ds;
        if (cudaSetDevice(ds->device) != cudaSuccess) { rc = set_error(RTP_ERR_CUDA, "cudaSetDevice"); break; }
        rc = ds->frame.reserve(npx * 4);
        if (rc == RTP_OK && samples_out) rc = ds->frame_samples.reserve(npx);
        d.ds = ds; d.st = ds->streams[0]; d.p = &frame[k].p;
        d.d_rgb = ds->frame.ptr;
        d.d_fg = foreground_out ? ds->frame.ptr + npx * 3 : nullptr;
        d.d_samples = samples_out ? ds->frame_samples.ptr : nullptr;
    }
    if (rc == RTP_OK) rc = render_adaptive(devs, camera, adaptive, stats != nullptr);
    for (size_t k = 0; k < devs.size() && rc == RTP_OK; ++k) {
        const AdaptiveDev& d = devs[k];
        cudaSetDevice(d.ds->device);
        rc = copy_rows(*d.p, d.st, {{rgb_out, d.d_rgb, 24}, {foreground_out, d.d_fg, 8}, {samples_out, d.d_samples, 4}});
    }
    return finish_frame(scene, frame, rc, stats, nullptr);
}

int rtp_render_adaptive_device(rtp_scene* scene, const rtp_camera* camera, const rtp_render_params* params, const rtp_adaptive_params* adaptive,
                               double* d_rgb_out, double* d_foreground_out, uint32_t* d_samples_out, rtp_stats* stats, void* cuda_stream) {
    if (!scene || !camera || !params || !adaptive || !d_rgb_out) return set_error(RTP_ERR_INVALID, "null argument");
    if (int rc = check_adaptive(params, adaptive)) return rc;
    std::vector<AdaptiveDev> devs(1);
    AdaptiveDev& d = devs[0];
    d.ds = scene->dev;
    std::lock_guard<std::mutex> guard(d.ds->lock);
    RTP_CUDA(cudaSetDevice(d.ds->device));
    d.st = static_cast<cudaStream_t>(cuda_stream);
    d.p = params;
    d.d_rgb = d_rgb_out; d.d_fg = d_foreground_out; d.d_samples = d_samples_out;
    int rc = render_adaptive(devs, camera, adaptive, stats != nullptr);
    const cudaError_t e = cudaStreamSynchronize(d.st);
    if (e != cudaSuccess && rc == RTP_OK) rc = set_error(RTP_ERR_CUDA, std::string("adaptive render: ") + cudaGetErrorString(e));
    if (rc == RTP_OK && stats) rc = render_finish(d.ds, stats);
    return rc;
}

}  // extern "C"
