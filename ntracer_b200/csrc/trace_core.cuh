// trace_core.cuh -- per-ray device code of the ntracer_b200 render path (sm_100a).
//
// Everything in here is written against the *semantics* of the reference's per-pixel path
// (Rouslan/NTracer src/tracer.hpp, cited per function as tracer.hpp:LINE) but shares none of its
// structure: the reference is recursive, pointer-based and heap-list-based; this is an explicit
// stack machine over a flat 16-byte-node arena with fixed-capacity per-ray lists, dimension as a
// template parameter (DT = 3..8) or run time (DT = 0), and the recursive colour evaluation
// linearised into RGB throughput weights so that reflection bounces can be deferred to wavefront
// queues (DESIGN.md section 4).
//
// The functions are __host__ __device__ so that tests/host_emul can run the very same state machine
// on the CPU against the oracle without a GPU.  That harness is test-only; the product .so contains
// only the __global__ kernels of kernels.cu and has no CPU path.
#pragma once
#include <float.h>
#include <math.h>
#include <stdint.h>

#include "device_types.h"

#if defined(__CUDACC__)
#define NTR_HD __host__ __device__ __forceinline__
#else
#define NTR_HD inline
#endif

// Loop unrolling policy of the translation unit: the fixed-dimension units (kern_d3..8.cu) unroll every
// per-component loop completely; the run-time-dimension unit (kern_dn.cu) defines NTR_GENERIC_UNIT and keeps
// them rolled (its trip counts are not compile-time constants and its vectors live in local memory).
#if defined(NTR_GENERIC_UNIT)
#define NTR_UNROLL _Pragma("unroll 1")
#else
#define NTR_UNROLL _Pragma("unroll")
#endif

namespace ntr {

#define NTR_FUZZ (FLT_EPSILON * 10)            /* ROUNDING_FUZZ, tracer.hpp:25 */
#define NTR_LIGHT_THRESHOLD (1.0f / 512)       /* tracer.hpp:31 */

template <int DT> struct DimCap { static constexpr int value = DT > 0 ? DT : NTR_MAXD; };
#define NTR_D(DT, s) (DT > 0 ? DT : (s).dim)

NTR_HD float ldf(const float *p) {
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}
NTR_HD uint32_t ldu(const uint32_t *p) {
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}
NTR_HD float4 ld4(const float *p) {
#if defined(__CUDA_ARCH__)
    return __ldg(reinterpret_cast<const float4 *>(p));
#else
    return *reinterpret_cast<const float4 *>(p);
#endif
}
NTR_HD uint2 lditem(const uint2 *p) {
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}
NTR_HD uint4 ldnode(const uint4 *p) {
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}
NTR_HD float rcp_approx(float x) {
#if defined(__CUDA_ARCH__)
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#else
    return 1.0f / x;
#endif
}
NTR_HD float u2f(uint32_t u) {
#if defined(__CUDA_ARCH__)
    return __uint_as_float(u);
#else
    float f; memcpy(&f, &u, 4); return f;
#endif
}
NTR_HD uint32_t f2u(float f) {
#if defined(__CUDA_ARCH__)
    return __float_as_uint(f);
#else
    uint32_t u; memcpy(&u, &f, 4); return u;
#endif
}

// v[i] with a run-time i: a select chain for compile-time D (stays in registers), plain indexing otherwise
template <int DT> NTR_HD float vsel(const float *v, int i) {
    if (DT > 0) {
        float r = v[0];
    NTR_UNROLL
        for (int k = 1; k < (DT > 0 ? DT : 1); ++k) r = (i == k) ? v[k] : r;
        return r;
    }
    return v[i];
}

struct Counters {
    unsigned long long node_steps = 0, simplex_tests = 0, solid_tests = 0, shadow_rays = 0, reflection_rays = 0,
                       shaded_hits = 0, truncated = 0;
};

struct Skip { uint32_t ref; int lane; };
struct HitRec { float dist; uint32_t ref; int lane; };

#ifndef NTR_BIG_SIMPLEX_PIPE
#define NTR_BIG_SIMPLEX_PIPE 1      // above 8 dimensions: simplex_single_big (vector loads, next edge requested ahead)
#endif

// ---- simplex records -------------------------------------------------------------------------------
// Register-staged view of one simplex record: stage 1 brings face_normal and d (enough for the plane
// test), stage 2 the rest.  DT == 0 reads through the pointer instead.
template <int DT> struct SimplexRec {
    static constexpr int S = (((DT + 1) * DT + 1) + 3) / 4 * 4;
    static constexpr int N1 = (DT + 1 + 3) / 4;
    // above 8 dimensions the record (>= 92 floats) is not staged in registers: stage 1 still brings face_normal and d
    // as float4s, the rest is read element by element where it is used (the edge loop exits early on most records)
    static constexpr bool STAGE_ALL = DT <= 8;
    float r[STAGE_ALL ? S : 4 * N1];
    const float *g;
    NTR_HD void stage1(const float *rec) {
        g = rec;
    NTR_UNROLL
        for (int k = 0; k < N1; ++k) {
            float4 v = ld4(rec + 4 * k);
            r[4 * k] = v.x; r[4 * k + 1] = v.y; r[4 * k + 2] = v.z; r[4 * k + 3] = v.w;
        }
    }
    NTR_HD void stage2() {
        if (STAGE_ALL) {
    NTR_UNROLL
            for (int k = N1; k < S / 4; ++k) {
                float4 v = ld4(g + 4 * k);
                r[4 * k] = v.x; r[4 * k + 1] = v.y; r[4 * k + 2] = v.z; r[4 * k + 3] = v.w;
            }
        }
    }
    NTR_HD float at(int i) const { return (STAGE_ALL || i < 4 * N1) ? r[i < (STAGE_ALL ? S : 4 * N1) ? i : 0] : ldf(g + i); }
    NTR_HD uint32_t meta(int sstride) const { return STAGE_ALL ? f2u(r[(STAGE_ALL ? S : 4 * N1) - 1]) : f2u(ldf(g + S - 1)); }
};
template <> struct SimplexRec<0> {
    const float *g;
    NTR_HD void stage1(const float *rec) { g = rec; }
    NTR_HD void stage2() {}
    NTR_HD float at(int i) const { return ldf(g + i); }
    NTR_HD uint32_t meta(int sstride) const { return f2u(ldf(g + sstride - 1)); }
};

// The single-simplex test above 8 dimensions, where the record (>= 92 floats) is not staged in registers as a whole.
// ncu, config 5 (1 M ten-dimensional simplexes, `profiles/r02_c5_ncu_full_summary.txt`): 68 % of the stall samples are
// long-scoreboard waits and 43 % of all samples sit on the edge loop, which read its 10 coefficients with scalar loads
// AFTER the previous edge's early-exit branch -- one trip to L1/L2 per edge on the dependency chain (the lanes of a warp
// are at different leaf items, so these are 20 different records per load instruction: L1 hit rate 59 %).  Here the
// record is read as aligned float4s: face normal, d and p1 in one batch (p1 no longer waits for the t test), and the
// float4s of edge e+1 are requested before edge e is evaluated.  Same arithmetic in the same order as simplex_single.
template <int DT>
NTR_HD float simplex_single_big(const SceneDev &s, uint32_t off, const float *o, const float *dir, float cutoff,
                                uint32_t &meta) {
    constexpr int D = DT;
    constexpr int S = (((DT + 1) * DT + 1) + 3) / 4 * 4;
    constexpr int E0 = 2 * D + 1;                   // first float of edge 0
    constexpr int NA = (E0 + 3) / 4;                // float4s that hold face_normal, d, p1
    constexpr int NW = (D + 2) / 4 + 1;             // float4s an edge of D floats can span
    const float *rec = s.simplex + off;
    float a[4 * NA];
#pragma unroll
    for (int k = 0; k < NA; ++k) {
        const float4 v = ld4(rec + 4 * k);
        a[4 * k] = v.x; a[4 * k + 1] = v.y; a[4 * k + 2] = v.z; a[4 * k + 3] = v.w;
    }
    float denom = 0, od = 0;
#pragma unroll
    for (int i = 0; i < D; ++i) { denom += a[i] * dir[i]; od += a[i] * o[i]; }
    if (denom == 0) return 0;
    const float t = -(od + a[D]) / denom;
    if (t <= 0 || t >= cutoff) return 0;
    float pside[D];
#pragma unroll
    for (int i = 0; i < D; ++i) pside[i] = a[D + 1 + i] - (o[i] + t * dir[i]);
    float cur[4 * NW], nxt[4 * NW];
#pragma unroll
    for (int k = 0; k < NW; ++k) {
        if (E0 / 4 + k <= (E0 + D - 1) / 4) {
            const float4 v = ld4(rec + 4 * (E0 / 4 + k));
            cur[4 * k] = v.x; cur[4 * k + 1] = v.y; cur[4 * k + 2] = v.z; cur[4 * k + 3] = v.w;
        }
    }
    float tot = 0;
#pragma unroll
    for (int e = 0; e < D - 1; ++e) {
        if (e + 1 < D - 1) {
            const int f0 = E0 + (e + 1) * D, q0 = f0 / 4, q1 = (f0 + D - 1) / 4;
#pragma unroll
            for (int k = 0; k < NW; ++k) {
                if (q0 + k <= q1) {
                    const float4 v = ld4(rec + 4 * (q0 + k));
                    nxt[4 * k] = v.x; nxt[4 * k + 1] = v.y; nxt[4 * k + 2] = v.z; nxt[4 * k + 3] = v.w;
                }
            }
        }
        const int base = (E0 + e * D) & 3;
        float area = 0;
#pragma unroll
        for (int i = 0; i < D; ++i) area += cur[base + i] * pside[i];
        if (area < -NTR_FUZZ || area > (1 + NTR_FUZZ)) return 0;
        tot += area;
#pragma unroll
        for (int k = 0; k < 4 * NW; ++k) cur[k] = nxt[k];
    }
    if (tot <= (1 + NTR_FUZZ)) { meta = f2u(ldf(rec + S - 1)); return t; }
    return 0;
}

// triangle::intersects (tracer.hpp:411-440): the single-primitive n-simplex test.  (The approximate-quotient pre-filter of
// batch_test was tried here too: config 5 got 3-4 % SLOWER -- one division per record is cheap next to the loads.)
template <int DT>
NTR_HD float simplex_single(const SceneDev &s, uint32_t off, const float *o, const float *dir, float cutoff,
                            uint32_t &meta) {
    if constexpr (DT > 8 && NTR_BIG_SIMPLEX_PIPE) return simplex_single_big<DT>(s, off, o, dir, cutoff, meta);
    const int D = NTR_D(DT, s);
    SimplexRec<DT> R;
    R.stage1(s.simplex + off);
    float denom = 0, od = 0;
    NTR_UNROLL
    for (int i = 0; i < D; ++i) { denom += R.at(i) * dir[i]; od += R.at(i) * o[i]; }
    if (denom == 0) return 0;
    float t = -(od + R.at(D)) / denom;
    if (t <= 0 || t >= cutoff) return 0;
    R.stage2();
    float pside[DimCap<DT>::value];
    NTR_UNROLL
    for (int i = 0; i < D; ++i) pside[i] = R.at(D + 1 + i) - (o[i] + t * dir[i]);
    float tot = 0;
    NTR_UNROLL
    for (int e = 0; e < D - 1; ++e) {
        float area = 0;
    NTR_UNROLL
        for (int i = 0; i < D; ++i) area += R.at(2 * D + 1 + e * D + i) * pside[i];
        if (area < -NTR_FUZZ || area > (1 + NTR_FUZZ)) return 0;
        tot += area;
    }
    if (tot <= (1 + NTR_FUZZ)) { meta = R.meta(s.sstride); return t; }
    return 0;
}

// Edge part of one batch lane (tracer.hpp:567-579): lower edge bound only, then the area sum.  The record is loaded
// into registers by load() AFTER the exact division of the plane test (issuing the loads before it was measured slower,
// round 1: config 2 0.746 -> 0.82 ms -- lanes rejected by the exact t test waste them).
template <int DT> struct EdgeRec {
    static constexpr int LP = DT > 0 ? (DT * DT + 3) / 4 * 4 : 4;
    static constexpr bool STAGED = DT > 0 && DT <= 8;          // see SimplexRec
    float r[STAGED ? LP : 4];
    const float *g;
    NTR_HD void load(const float *lp) {
        g = lp;
        if (STAGED) {
    NTR_UNROLL
            for (int k = 0; k < LP / 4; ++k) {
                const float4 v = ld4(lp + 4 * k);
                r[4 * k] = v.x; r[4 * k + 1] = v.y; r[4 * k + 2] = v.z; r[4 * k + 3] = v.w;
            }
        }
    }
    NTR_HD float at(int k) const { return STAGED ? r[k < (STAGED ? LP : 4) ? k : 0] : ldf(g + k); }
};

template <int DT>
NTR_HD bool batch_lane_edges(const SceneDev &s, const EdgeRec<DT> &er, const float *o, const float *dir, float t) {
    const int D = NTR_D(DT, s);
    float pside[DimCap<DT>::value];
    NTR_UNROLL
    for (int i = 0; i < D; ++i) pside[i] = er.at(i) - (o[i] + t * dir[i]);
    float tot = 0;
    NTR_UNROLL
    for (int e = 0; e < D - 1; ++e) {
        float area = 0;
    NTR_UNROLL
        for (int i = 0; i < D; ++i) area += er.at(D + e * D + i) * pside[i];
        if (!(area >= -NTR_FUZZ)) return false;
        tot += area;
    }
    return tot <= (1 + NTR_FUZZ);
}

// triangle_batch::intersects (tracer.hpp:551-599) over a batch block (arena_pack.h): per group of 4 lanes the
// plane test runs on SoA float4s (t >= 0 mask, :561-565); lanes that can still beat the running minimum go
// through the edge part; the winner is the lowest lane with the strictly smallest t (:583-594).
template <int DT, int FLAGS>
NTR_HD float batch_test(const SceneDev &s, uint32_t off, const float *o, const float *dir, int &index, float cutoff,
                        uint32_t &meta, Counters &cnt) {
    const int D = NTR_D(DT, s);
    // fixed-dimension kernels are only used with 4-lane batches (the host routes anything else to the run-time
    // dimension kernels), which makes every address below a compile-time offset from `blk`
    const int B = DT > 0 ? 4 : s.batch;
    const int LPART = DT > 0 ? (DT * DT + 3) / 4 * 4 : s.lane_part;
    const float *blk = s.batches + off;
    const float *edges = blk + (D + 1) * B;
    float min_t = cutoff;
    int r_index = -1;
    for (int g = 0; g < B; g += 4) {
        float den[4] = {0, 0, 0, 0}, od[4] = {0, 0, 0, 0};
    NTR_UNROLL
        for (int i = 0; i < D; ++i) {
            const float4 f = ld4(blk + i * B + g);
            den[0] += f.x * dir[i]; den[1] += f.y * dir[i]; den[2] += f.z * dir[i]; den[3] += f.w * dir[i];
            od[0] += f.x * o[i]; od[1] += f.y * o[i]; od[2] += f.z * o[i]; od[3] += f.w * o[i];
        }
        const float4 dd = ld4(blk + D * B + g);
        const float dv[4] = {dd.x, dd.y, dd.z, dd.w};
        float num[4];
        unsigned viable = 0;
        // Pre-filter with an approximate quotient (MUFU.RCP + FMUL instead of an IEEE division per lane).  It only
        // ever REJECTS lanes the exact test below would reject as well: the approximate quotient is within 2^-21
        // of the correctly rounded one (normal-range denominators only), its sign is exact, and the cutoff
        // comparison leaves a 2^-20 margin; everything else falls through to the exact division.
        const float cut = min_t * 1.000001f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            num[k] = -(od[k] + dv[k]);
            const float ta = num[k] * rcp_approx(den[k]);
            const bool reject = (fabsf(den[k]) > 1e-30f) & ((ta < 0) | (ta > cut));
            viable |= ((reject | (g + k == index)) ? 0u : 1u) << k;
        }
        if (FLAGS & NTR_F_COUNT) cnt.simplex_tests += 4;
        if (!viable) continue;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (!(viable & (1u << k))) continue;
            if (den[k] == 0) continue;
            // mask = denom != 0 && t >= 0 (:562-565); t[i] && t[i] < min_t (:586)
            EdgeRec<DT> er;
            const float t = num[k] / den[k];
            if (!(t >= 0) || t == 0 || !(t < min_t)) continue;
            er.load(edges + (g + k) * LPART);
            if (!batch_lane_edges<DT>(s, er, o, dir, t)) continue;
            min_t = t;
            r_index = g + k;
        }
    }
    if (r_index == -1) return 0;
    index = r_index;
    meta = f2u(ldf(edges + B * LPART + r_index));
    return min_t;
}

// Geometry of a simplex hit: normal.origin = o + t*dir, normal.direction = +-unit(face_normal)
// (tracer.hpp:434-436, 595-597).
template <int DT>
NTR_HD void simplex_normal(const SceneDev &s, uint32_t idx, const float *o, const float *dir, float t, float *P,
                           float *N) {
    const int D = NTR_D(DT, s);
    const float *rec = s.simplex + (size_t)idx * s.sstride;
    float fn[DimCap<DT>::value];
    float denom = 0, sq = 0;
    NTR_UNROLL
    for (int i = 0; i < D; ++i) { fn[i] = ldf(rec + i); denom += fn[i] * dir[i]; sq += fn[i] * fn[i]; }
    float len = sqrtf(sq);
    NTR_UNROLL
    for (int i = 0; i < D; ++i) {
        P[i] = o[i] + t * dir[i];
        float u = fn[i] / len;
        N[i] = denom > 0 ? -u : u;
    }
}

// ---- solids ----------------------------------------------------------------------------------------
// solid::intersects (tracer.hpp:251-276) with hypercube_intersects (:126-152) / hypersphere_intersects
// (:154-173).  P/N receive what the reference writes into `normal`; `wmask` has a bit per component of
// normal.origin that was written (the cube test writes local-space coordinates into it even when it
// misses -- DESIGN.md section 4, quirk Q12).
template <int DT>
NTR_HD float solid_test(const SceneDev &s, uint32_t idx, const float *o, const float *dir, float cutoff, float *P,
                        float *N, uint32_t &wmask, uint32_t &meta) {
    const int D = NTR_D(DT, s);
    const float *rec = s.solids + (size_t)idx * s.solstride;
    const int type = (int)ldf(rec);
    const float *inv = rec + 1, *pos = rec + 1 + D * D, *orient = rec + 1 + D * D + D;
    float to[DimCap<DT>::value], td[DimCap<DT>::value];
    NTR_UNROLL
    for (int i = 0; i < D; ++i) {
        float a = 0, b = 0;
    NTR_UNROLL
        for (int j = 0; j < D; ++j) { float m = ldf(inv + i * D + j); a += m * o[j]; b += m * dir[j]; }
        to[i] = a - ldf(pos + i);
        td[i] = b;
    }
    wmask = 0;
    float dist = 0;
    float ln[DimCap<DT>::value];      // local-space normal.direction
    if (type == NTR_SOLID_CUBE) {
        bool found = false;
        for (int i = 0; i < D && !found; ++i) {
            float di = vsel<DT>(td, i);
            if (di != 0) {
                float face = di < 0 ? 1.0f : -1.0f;
                float dd = (face - vsel<DT>(to, i)) / di;
    NTR_UNROLL
                for (int k = 0; k < D; ++k) if (k == i) P[k] = face;
                wmask |= 1u << i;
                if (dd > 0) {
                    bool miss = false;
    NTR_UNROLL
                    for (int j = 0; j < D; ++j) {
                        if (!miss && j != i) {
                            float v = td[j] * dd + to[j];
                            P[j] = v;
                            wmask |= 1u << j;
                            if (fabsf(v) > (1 + NTR_FUZZ)) miss = true;
                        }
                    }
                    if (!miss) {
                        if (dd >= cutoff) return 0;
    NTR_UNROLL
                        for (int k = 0; k < D; ++k) ln[k] = (k == i) ? face : 0.0f;
                        dist = dd;
                        found = true;
                    }
                }
            }
        }
        if (!found) return 0;
    } else {
        float a = 0, b = 0, c = 0;
    NTR_UNROLL
        for (int i = 0; i < D; ++i) { a += td[i] * td[i]; b += td[i] * to[i]; c += to[i] * to[i]; }
        b = 2 * b;
        c = c - 1;
        float disc = b * b - 4 * a * c;
        if (disc < 0) return 0;
        float dd = (-b - sqrtf(disc)) / (2 * a);
        if (dd <= 0 || dd >= cutoff) return 0;
    NTR_UNROLL
        for (int i = 0; i < D; ++i) { P[i] = to[i] + td[i] * dd; ln[i] = P[i]; }
        dist = dd;
    }
    // back-transform (tracer.hpp:273-274): origin = orientation*(origin + position), direction = orientation*direction
    float tmp[DimCap<DT>::value];
    NTR_UNROLL
    for (int i = 0; i < D; ++i) tmp[i] = P[i] + ldf(pos + i);
    NTR_UNROLL
    for (int i = 0; i < D; ++i) {
        float a = 0, b = 0;
    NTR_UNROLL
        for (int j = 0; j < D; ++j) { float m = ldf(orient + i * D + j); a += m * tmp[j]; b += m * ln[j]; }
        P[i] = a;
        N[i] = b;
    }
    wmask = 0xFFFFFFFFu;
    meta = f2u(ldf(rec + s.solstride - 1));
    return dist;
}

// material index / opacity bit of a hit target
template <int DT> NTR_HD uint32_t target_meta(const SceneDev &s, uint32_t ref, int lane) {
    uint32_t kind = ref >> 30, idx = ref & NTR_IDX_MASK;
    if (kind == NTR_REF_SOLID) return f2u(ldf(s.solids + (size_t)idx * s.solstride + s.solstride - 1));
    if (kind == NTR_REF_BATCH) idx += (uint32_t)lane;
    return f2u(ldf(s.simplex + (size_t)idx * s.sstride + s.sstride - 1));
}
NTR_HD int flat_prim_id(const SceneDev &s, uint32_t ref, int lane) {
    uint32_t kind = ref >> 30, idx = ref & NTR_IDX_MASK;
    if (kind == NTR_REF_BATCH) return (int)(idx + (uint32_t)lane);
    if (kind == NTR_REF_SIMPLEX) return (int)idx;
    return (int)(s.n_simplex + idx);
}

// ---- per-ray lists of the general variant -------------------------------------------------------------
struct HitList {                        // quick_list<ray_intersection>, tracer.hpp:663-729,781
    float dist[NTR_THITS_CAP];
    uint32_t ref[NTR_THITS_CAP];
    signed char lane[NTR_THITS_CAP];
    int n;
    int dropped;
    NTR_HD void clear() { n = 0; dropped = 0; }
    NTR_HD void add(float d, uint32_t r, int l) {
        if (n < NTR_THITS_CAP) { dist[n] = d; ref[n] = r; lane[n] = (signed char)l; ++n; }
        else dropped = 1;
    }
    // trim_intersections (tracer.hpp:784-789) with quick_list::remove_at's swap-with-last (:723-728)
    NTR_HD void trim(float d, int from) {
        while (from < n) {
            if (dist[from] >= d) {
                --n;
                if (from != n) { dist[from] = dist[n]; ref[from] = ref[n]; lane[from] = lane[n]; }
            } else ++from;
        }
    }
    // sort_and_unique (tracer.hpp:714-721): by distance, then drop adjacent entries with the same target
    NTR_HD void sort_and_unique() {
        for (int i = 1; i < n; ++i) {
            float d = dist[i]; uint32_t r = ref[i]; signed char l = lane[i];
            int j = i;
            while (j > 0 && d < dist[j - 1]) { dist[j] = dist[j - 1]; ref[j] = ref[j - 1]; lane[j] = lane[j - 1]; --j; }
            dist[j] = d; ref[j] = r; lane[j] = l;
        }
        if (n == 0) return;
        int w = 0;
        for (int i = 1; i < n; ++i) {
            if (!(ref[i] == ref[w] && lane[i] == lane[w])) {
                ++w;
                dist[w] = dist[i]; ref[w] = ref[i]; lane[w] = lane[i];
            }
        }
        n = w + 1;
    }
};

// The exact mailbox of scenes with big leaves.  The reference's `checked` list (tracer.hpp:782,832-834) answers "was this
// item tested during this traversal" for every item; its implementation breaks beyond 20 entries (quick_list growth
// copies bytes, :670-680), the oracle restates it with a correct unbounded list.  On the star polytopes a leaf alone
// holds up to 1,600 items and every batch sits in ~80 leaves, so a bounded table is overrun at once and the same
// batches are tested again in leaf after leaf (host emulation, {5/2,3,3}: 1,318 simplex tests per pixel against the
// oracle's 764).  Here every traversing thread owns one bit per leaf item in a scene-wide table in device memory
// (column-interleaved: word w of thread t at [w * threads + t], so that the lanes of a warp of coherent rays, which
// test the same item at the same time, touch one 128-byte line).  Words carry an 8-bit generation tag, so starting a
// new traversal costs one increment instead of clearing the column; a word written by an older traversal reads as
// empty.  This is the oracle's semantics exactly -- pixels beyond the reference's own limit included.
struct MailboxStore {
    uint32_t *col;          // this thread's column (nullptr: the scene has none -> bounded table)
    uint32_t stride;        // threads in the table
    uint32_t words;         // words per thread
    uint32_t gen;           // generation of the current traversal, 1..255
    uint32_t solid_base;    // key of solid 0
    uint32_t shift;         // SceneDev::mb_shift
    // bind to thread `tid` of the scene's table; the generation counter of the column survives between launches in the
    // word behind its bit words (a column starts all zero: generation 0 is never current)
    NTR_HD void attach(uint32_t *table, uint32_t n_words, uint32_t n_threads, uint32_t tid, uint32_t n_simplex, uint32_t key_shift) {
        col = (table && tid < n_threads) ? table + tid : nullptr;
        stride = n_threads; words = n_words; shift = key_shift; solid_base = (n_simplex >> key_shift) + 1;
        gen = col ? col[(size_t)words * stride] : 0u;
    }
    NTR_HD void detach() { if (col) col[(size_t)words * stride] = gen; }
    NTR_HD void begin_traversal() {
        if (++gen > 255u) {
            for (uint32_t w = 0; w < words; ++w) col[(size_t)w * stride] = 0u;
            gen = 1u;
        }
    }
    // The queries take the table's geometry from the scene constants (kernel parameters: constant-bank operands) and the
    // column / generation by value: ncu, config 4, showed this descriptor being re-read from local memory field by field
    // on every item of every leaf (a fifth of the kernel's local-memory instructions).
    NTR_HD static uint32_t key_of(const SceneDev &s, uint32_t r) {
        return (r >> 30) == NTR_REF_SOLID ? (s.n_simplex >> s.mb_shift) + 1u + (r & NTR_IDX_MASK) : (r & NTR_IDX_MASK) >> s.mb_shift;
    }
    NTR_HD static bool has(const SceneDev &s, const uint32_t *col, uint32_t gen, uint32_t r) {
        const uint32_t k = key_of(s, r), w = col[(size_t)(k / NTR_MAILBOX_BITS_PER_WORD) * s.mb_threads];
        return (w >> 24) == gen && ((w >> (k % NTR_MAILBOX_BITS_PER_WORD)) & 1u);
    }
    NTR_HD static void add(const SceneDev &s, uint32_t *col, uint32_t gen, uint32_t r) {
        const uint32_t k = key_of(s, r);
        uint32_t *p = col + (size_t)(k / NTR_MAILBOX_BITS_PER_WORD) * s.mb_threads;
        const uint32_t w = *p;
        *p = ((w >> 24) == gen ? w : gen << 24) | (1u << (k % NTR_MAILBOX_BITS_PER_WORD));
    }
};

struct Mailbox {                        // prim_list `checked`, tracer.hpp:782,832-834
    // The reference's list is defined up to 20 entries (quick_list growth copies bytes, tracer.hpp:670-680: beyond
    // that has() scans uninitialised slots).  This one is exact up to NTR_MAILBOX_CAP entries and then switches itself
    // off -- in that regime the reference skips primitives at random, so there is nothing left to be faithful to, and
    // a membership test per item of a 1,600-item leaf would dominate the frame.
    // Only membership matters (the reference scans its list linearly, :832-834), so the entries live in a small
    // open-addressing table: one or two probes per query instead of up to 40 compares (ncu, config 4, round 2: the
    // linear scan was 16 % of all executed instructions and a quarter of the local-memory traffic of the kernel).
    uint32_t v[NTR_MAILBOX_SLOTS];      // NTR_NONE_REF = empty slot (no item ref has both type bits set)
    int n;
    MailboxStore *big;                  // set: the exact per-thread bitset replaces the table (scenes with big leaves)
    uint32_t *col;                      // ... its column and the generation of the traversal in progress, by value
    uint32_t gen;
    static_assert((NTR_MAILBOX_SLOTS & (NTR_MAILBOX_SLOTS - 1)) == 0 && NTR_MAILBOX_SLOTS > NTR_MAILBOX_CAP, "mailbox table size");
    NTR_HD static uint32_t slot_of(uint32_t r) { return (r * 2654435761u) >> 16 & (uint32_t)(NTR_MAILBOX_SLOTS - 1); }
    NTR_HD bool exact() const { return big != nullptr; }
    NTR_HD void clear() {
        n = 0;
        if (big) { big->begin_traversal(); col = big->col; gen = big->gen; return; }
        for (int i = 0; i < NTR_MAILBOX_SLOTS; ++i) v[i] = NTR_NONE_REF;
    }
    NTR_HD bool has(const SceneDev &s, uint32_t r) const {
        if (big) return MailboxStore::has(s, col, gen, r);
        if (n > NTR_MAILBOX_CAP || n == 0) return false;
        uint32_t h = slot_of(r);
        for (;;) {
            const uint32_t x = v[h];
            if (x == r) return true;
            if (x == NTR_NONE_REF) return false;
            h = (h + 1) & (uint32_t)(NTR_MAILBOX_SLOTS - 1);
        }
    }
    NTR_HD void add(const SceneDev &s, uint32_t r) {
        if (big) { MailboxStore::add(s, col, gen, r); return; }
        if (n < NTR_MAILBOX_CAP) {
            uint32_t h = slot_of(r);
            while (v[h] != NTR_NONE_REF) h = (h + 1) & (uint32_t)(NTR_MAILBOX_SLOTS - 1);
            v[h] = r;
            ++n;
        } else n = NTR_MAILBOX_CAP + 1;
    }
};

template <int DT> struct GenState {
    float hitP[DimCap<DT>::value], hitN[DimCap<DT>::value];    // o_hit.normal as the reference leaves it
    HitList th;
    Mailbox mb;
};

// Per-ray constants of the traversal.
template <int DT> struct RaySlab {
    float invdir[DimCap<DT>::value];
    NTR_HD void init(const SceneDev &s, const float *dir) {
        const int D = NTR_D(DT, s);
    NTR_UNROLL
        for (int i = 0; i < D; ++i) invdir[i] = 1 / dir[i];      // tracer.hpp:1174
    }
};

// ---- leaves ----------------------------------------------------------------------------------------
// kd_leaf::intersects for all-opaque, simplex-only scenes.  Without transparent hits and solids the
// reference's mailbox, two-phase loop and final trim (tracer.hpp:977-1086) cannot influence the result:
// a re-tested primitive misses its own cutoff, so only the running nearest hit matters.
// Small per-traversal mailbox of the opaque variant: purely an optimisation (a batch that was already tested against
// this ray can only miss its own cutoff again, see above), so false negatives are harmless.  The NTR_MINI_MAILBOX
// most recently tested batch refs, kept as a shift register (0 = disabled).  Measured on config 2: 8 entries
// remove 35 % of the simplex tests, 16 remove 42 % (the reference's unbounded list removes 39 %); 8 entries at 64
// registers / 8 CTAs per SM beat 16 entries at 80 registers / 6 CTAs (config 2 -3.5 %, config 4 opaque -10 %).
// (Measured and dropped, round 1 / round 2: testing two batch items per iteration, 34.6 -> 38.7 ms on config 4 opaque;
// prefetching the next item's record; a direct-mapped per-ray table for single simplexes in local memory, config 5
// reduced 23.2 -> 23.7 ms with 64 entries, 24.9 ms with 256.)
#ifndef NTR_MINI_MAILBOX
#define NTR_MINI_MAILBOX 8
#endif
struct MiniMailbox {
#if NTR_MINI_MAILBOX > 0
    uint32_t v[NTR_MINI_MAILBOX];       // most recent first; constant indices only, so it lives in registers
    NTR_HD void clear() {
#pragma unroll
        for (int i = 0; i < NTR_MINI_MAILBOX; ++i) v[i] = NTR_NONE_REF;
    }
    NTR_HD bool test_and_set(uint32_t r) {
        bool f = false;
#pragma unroll
        for (int i = 0; i < NTR_MINI_MAILBOX; ++i) f |= v[i] == r;
        if (!f) {
#pragma unroll
            for (int i = NTR_MINI_MAILBOX - 1; i > 0; --i) v[i] = v[i - 1];
            v[0] = r;
        }
        return f;
    }
#else
    NTR_HD void clear() {}
    NTR_HD bool test_and_set(uint32_t) { return false; }
#endif
};

template <int DT, int FLAGS>
NTR_HD bool leaf_opaque(const SceneDev &s, const uint4 node, const float *o, const float *dir, const RaySlab<DT> &rs,
                        Skip skip, HitRec &oh, MiniMailbox &mm, Counters &cnt) {
    const uint2 *items = s.leaf_items + node.y;
    const uint32_t size = node.z;
    bool hit = false;
    for (uint32_t i = 0; i < size; ++i) {
        const uint2 it = lditem(items + i);
        const uint32_t item = it.x;
        uint32_t meta;
        if ((item >> 30) == NTR_REF_BATCH) {
            if (mm.test_and_set(item)) continue;
            int index = skip.ref == item ? skip.lane : -1;
            float dist = batch_test<DT, FLAGS>(s, it.y, o, dir, index, oh.dist, meta, cnt);
            if (dist) { oh.dist = dist; oh.ref = item; oh.lane = index; hit = true; }
        } else if (item != skip.ref) {
            if (FLAGS & NTR_F_COUNT) cnt.simplex_tests++;
            float dist = simplex_single<DT>(s, it.y, o, dir, oh.dist, meta);
            if (dist) { oh.dist = dist; oh.ref = item; oh.lane = -1; hit = true; }
        }
    }
    return hit;
}

// One primitive test of the general variant; P/N/wmask as in solid_test.
template <int DT, int FLAGS>
NTR_HD float prim_test_general(const SceneDev &s, uint2 it, const float *o, const float *dir, float cutoff,
                               Skip skip, int &lane, float *P, float *N, uint32_t &wmask, uint32_t &meta,
                               Counters &cnt) {
    const uint32_t item = it.x, off = it.y;
    const uint32_t kind = item >> 30, idx = item & NTR_IDX_MASK;
    wmask = 0;
    float dist;
    if (kind == NTR_REF_BATCH) {
        lane = skip.ref == item ? skip.lane : -1;
        dist = batch_test<DT, FLAGS>(s, off, o, dir, lane, cutoff, meta, cnt);
        if (dist) { simplex_normal<DT>(s, idx + (uint32_t)lane, o, dir, dist, P, N); wmask = 0xFFFFFFFFu; }
    } else if (kind == NTR_REF_SIMPLEX) {
        lane = -1;
        if (FLAGS & NTR_F_COUNT) cnt.simplex_tests++;
        dist = simplex_single<DT>(s, off, o, dir, cutoff, meta);
        if (dist) { simplex_normal<DT>(s, idx, o, dir, dist, P, N); wmask = 0xFFFFFFFFu; }
    } else {
        lane = -1;
        if (FLAGS & NTR_F_COUNT) cnt.solid_tests++;
        dist = solid_test<DT>(s, idx, o, dir, cutoff, P, N, wmask, meta);
    }
    return dist;
}

// The count of the `goto hit` re-test of an item that gave the first opaque hit of a leaf (below): the test always misses
// its own cutoff, so it is counted, not run.  The item-by-item scan and the chunked replay count it alike.
template <int DT, int FLAGS>
NTR_HD void count_retest(const SceneDev &s, uint32_t item, Counters &cnt) {
    if (FLAGS & NTR_F_COUNT) {
        if ((item >> 30) == NTR_REF_SOLID) cnt.solid_tests++;
        else cnt.simplex_tests += (item >> 30) == NTR_REF_BATCH ? (uint32_t)(((DT > 0 ? 4 : s.batch) + 3) / 4 * 4) : 1u;
    }
}

// kd_leaf<Store,true>::intersects (tracer.hpp:977-1086), every observable behaviour kept:
//   phase 0 (before the first opaque hit of this leaf): tests write straight into o_hit.normal;
//   the first opaque hit switches to phase 1 WITHOUT marking the item checked, so the same item is
//   tested again (and misses its own cutoff); in phase 1 a closer opaque hit replaces o_hit;
//   finally transparent hits of this leaf at or beyond the LAST test's result are dropped.
template <int DT, int FLAGS>
NTR_HD bool leaf_general(const SceneDev &s, const uint4 node, const float *o, const float *dir, const RaySlab<DT> &rs,
                         Skip skip, HitRec &oh, GenState<DT> &g, Counters &cnt) {
    const int D = NTR_D(DT, s);
    const uint2 *items = s.leaf_items + node.y;
    const uint32_t size = node.z;
    const int h_start = g.th.n;
    float dist = 0;
    bool phase1 = false;
    float P[DimCap<DT>::value], N[DimCap<DT>::value];
    for (uint32_t i = 0; i < size; ++i) {
        const uint2 it = lditem(items + i);
        const uint32_t item = it.x;
        const bool is_batch = (item >> 30) == NTR_REF_BATCH;
        if ((!is_batch && item == skip.ref) || g.mb.has(s, item)) continue;
        int lane;
        uint32_t wmask, meta;
        dist = prim_test_general<DT, FLAGS>(s, it, o, dir, oh.dist, skip, lane, P, N, wmask, meta, cnt);
        if (!phase1) {
            if (wmask) {
    NTR_UNROLL
                for (int k = 0; k < D; ++k) if (wmask & (1u << k)) g.hitP[k] = P[k];
            }
            if (dist) {
    NTR_UNROLL
                for (int k = 0; k < D; ++k) g.hitN[k] = N[k];
                if (meta & NTR_META_OPAQUE) {
                    oh.dist = dist; oh.ref = item; oh.lane = lane;
                    phase1 = true;
                    // `goto hit` tests this item once more before it is marked checked (tracer.hpp:1008,1041).  With the
                    // cutoff now at its own distance that test can only miss (the comparison is strict, the arithmetic the
                    // same) and a miss in phase 1 writes nothing: what it leaves behind is the last-test result 0 (Q13)
                    // and its count.
                    dist = 0;
                    count_retest<DT, FLAGS>(s, item, cnt);
                } else {
                    g.th.add(dist, item, lane);
                }
            }
        } else if (dist) {
            if (meta & NTR_META_OPAQUE) {
                oh.dist = dist; oh.ref = item; oh.lane = lane;
    NTR_UNROLL
                for (int k = 0; k < D; ++k) { g.hitP[k] = P[k]; g.hitN[k] = N[k]; }
            } else {
                g.th.add(dist, item, lane);
            }
        }
        g.mb.add(s, item);
    }
    if (!phase1) return false;
    g.th.trim(dist, h_start);           // `dist`: the result of the last test (Q3)
    return true;
}

// ---- chunked evaluation of a leaf (general variant) -------------------------------------------------------------
// What lets ONE ray's scan of a big leaf be split over the lanes of a warp (trace_warp.cuh; DESIGN.md section 4: a single
// ray through the 1,600-item leaves of {5/2,3,3} is what bounds a frame once the bulk is spread thin).  The leaf is cut
// into chunks; all tests of a chunk are evaluated against the state at the START of the chunk (that is the part 32 lanes
// can do at once), then their results are REPLAYED in leaf order with the sequential semantics of kd_leaf::intersects.
// Exactness of the replay:
//   * a test run with the looser cutoff of the chunk start returns, for simplexes, batches and spheres, either the same
//     hit the tighter cutoff would give or a hit at t >= the tighter cutoff, which the replay demotes to a miss (a batch
//     reports the lowest lane with the smallest t, which does not depend on the cutoff as long as it passes it);
//   * hypercubes write partial local-space coordinates into o_hit.normal before they compare with the cutoff (Q12), so
//     a demoted hypercube hit is simply tested again with the current cutoff (rare);
//   * the mailbox can only change its answer for an item of the chunk by switching itself off (overflow) in the
//     middle of it; an item skipped at evaluation time but no longer skipped at replay time is tested on the spot;
//   * the re-test after the first opaque hit (`goto hit`, Q13) always misses its own cutoff: the replay records a miss.
// leaf_general_chunked below evaluates the chunk in a loop on one thread; it exists so that the replay logic is proven
// against the oracle in the CPU tier (host emulation, -DNTR_CHUNKED_LEAVES=1, tests/test_fuzz_emul.py).
#ifndef NTR_CHUNKED_LEAVES
#define NTR_CHUNKED_LEAVES 0
#endif
// warp-synchronous code exists on the device, and on the host when the test harness emulates a warp with 32 threads
// (tests/host_emul/emul.cpp, -DNTR_EMULATE_WARP)
#if defined(__CUDACC__) || defined(NTR_EMULATE_WARP)
#define NTR_WARP_CODE 1
#else
#define NTR_WARP_CODE 0
#endif
#ifndef NTR_CHUNK
#define NTR_CHUNK 32
#endif
#ifndef NTR_CHUNK_LEAF_MIN
#define NTR_CHUNK_LEAF_MIN 1
#endif
template <int DT> struct ChunkEval {
    float dist;
    int lane;
    uint32_t wmask, meta;
    bool skipped;
    bool geom;          // P / N hold what the test wrote (always for solids; simplex hits may leave it to the replay)
    float P[DimCap<DT>::value], N[DimCap<DT>::value];
};

// One primitive test of the general variant without the hit geometry of simplexes (the replay computes it for the
// hits that survive): what a lane of a cooperating warp evaluates.
template <int DT, int FLAGS>
NTR_HD void prim_eval(const SceneDev &s, uint2 it, const float *o, const float *dir, float cutoff, Skip skip,
                      ChunkEval<DT> &e, Counters &cnt) {
    const uint32_t item = it.x, off = it.y;
    const uint32_t kind = item >> 30;
    e.wmask = 0; e.meta = 0; e.geom = false; e.skipped = false;
    if (kind == NTR_REF_BATCH) {
        e.lane = skip.ref == item ? skip.lane : -1;
        e.dist = batch_test<DT, FLAGS>(s, off, o, dir, e.lane, cutoff, e.meta, cnt);
    } else if (kind == NTR_REF_SIMPLEX) {
        e.lane = -1;
        if (FLAGS & NTR_F_COUNT) cnt.simplex_tests++;
        e.dist = simplex_single<DT>(s, off, o, dir, cutoff, e.meta);
    } else {
        e.lane = -1;
        if (FLAGS & NTR_F_COUNT) cnt.solid_tests++;
        e.dist = solid_test<DT>(s, item & NTR_IDX_MASK, o, dir, cutoff, e.P, e.N, e.wmask, e.meta);
        e.geom = true;
    }
}

// One step of the replay: what kd_leaf::intersects does with the test of one item, given the result `e` of that test
// taken earlier (with a cutoff that may have been looser, and before the mailbox may have switched itself off).
template <int DT, int FLAGS>
NTR_HD void replay_item(const SceneDev &s, const uint2 it, const float *o, const float *dir, Skip skip, HitRec &oh,
                        GenState<DT> &g, Counters &cnt, bool &phase1, float &dist, ChunkEval<DT> &e,
                        bool mailbox_done = false /* the caller consulted and updated the mailbox for this item */) {
    const int D = NTR_D(DT, s);
    const uint32_t item = it.x;
    const bool is_batch = (item >> 30) == NTR_REF_BATCH;
    if ((!is_batch && item == skip.ref) || (!mailbox_done && g.mb.has(s, item))) return;
    const bool stale_cutoff = e.dist != 0 && !(e.dist < oh.dist);
    const bool is_cube = (item >> 30) == NTR_REF_SOLID &&
                         (int)ldf(s.solids + (size_t)(item & NTR_IDX_MASK) * s.solstride) == NTR_SOLID_CUBE;
    if (e.skipped || (stale_cutoff && is_cube)) {
        e.dist = prim_test_general<DT, FLAGS>(s, it, o, dir, oh.dist, skip, e.lane, e.P, e.N, e.wmask, e.meta, cnt);
        e.geom = true;
    } else if (stale_cutoff) {
        e.dist = 0;             // simplexes and spheres leave o_hit.normal alone when they miss
        e.wmask = 0;
    }
    dist = e.dist;
    if (dist && !e.geom) {      // a simplex hit evaluated without its geometry (prim_eval)
        simplex_normal<DT>(s, (item & NTR_IDX_MASK) + (is_batch ? (uint32_t)e.lane : 0u), o, dir, dist, e.P, e.N);
        e.wmask = 0xFFFFFFFFu;
        e.geom = true;
    }
    if (!phase1) {
    NTR_UNROLL
        for (int k = 0; k < D; ++k) if (e.wmask & (1u << k)) g.hitP[k] = e.P[k];
        if (dist) {
    NTR_UNROLL
            for (int k = 0; k < D; ++k) g.hitN[k] = e.N[k];
            if (e.meta & NTR_META_OPAQUE) {
                oh.dist = dist; oh.ref = item; oh.lane = e.lane;
                phase1 = true;
                dist = 0;       // the re-test of `goto hit` misses its own cutoff (and then the item is added)
                count_retest<DT, FLAGS>(s, item, cnt);
            } else {
                g.th.add(dist, item, e.lane);
            }
        }
    } else if (dist) {
        if (e.meta & NTR_META_OPAQUE) {
            oh.dist = dist; oh.ref = item; oh.lane = e.lane;
    NTR_UNROLL
            for (int k = 0; k < D; ++k) { g.hitP[k] = e.P[k]; g.hitN[k] = e.N[k]; }
        } else {
            g.th.add(dist, item, e.lane);
        }
    }
    if (!mailbox_done) g.mb.add(s, item);
}

template <int DT, int FLAGS>
NTR_HD bool leaf_general_chunked(const SceneDev &s, const uint4 node, const float *o, const float *dir, const RaySlab<DT> &rs,
                                 Skip skip, HitRec &oh, GenState<DT> &g, Counters &cnt) {
    const uint2 *items = s.leaf_items + node.y;
    const uint32_t size = node.z;
    const int h_start = g.th.n;
    float dist = 0;
    bool phase1 = false;
    ChunkEval<DT> ev[NTR_CHUNK];
    for (uint32_t base = 0; base < size; base += NTR_CHUNK) {
        const uint32_t n = size - base < NTR_CHUNK ? size - base : NTR_CHUNK;
        // ---- evaluation: every item of the chunk against the cutoff and the mailbox as they are now ----
        const float cutoff0 = oh.dist;
        for (uint32_t j = 0; j < n; ++j) {
            const uint2 it = lditem(items + base + j);
            const bool is_batch = (it.x >> 30) == NTR_REF_BATCH;
            const bool skipped = (!is_batch && it.x == skip.ref) || g.mb.has(s, it.x);
            ev[j].dist = 0; ev[j].wmask = 0; ev[j].meta = 0; ev[j].lane = -1; ev[j].geom = false;
            if (!skipped) prim_eval<DT, FLAGS>(s, it, o, dir, cutoff0, skip, ev[j], cnt);
            ev[j].skipped = skipped;
        }
        // ---- replay in leaf order ----
        for (uint32_t j = 0; j < n; ++j)
            replay_item<DT, FLAGS>(s, lditem(items + base + j), o, dir, skip, oh, g, cnt, phase1, dist, ev[j]);
    }
    if (!phase1) return false;
    g.th.trim(dist, h_start);
    return true;
}

// Per-ray axis tables of the traversal.  A k-d step needs o[axis], dir[axis] and 1/dir[axis] for a run-time axis; with
// the vectors in registers that is a select chain per value -- 3 x (D-1) selects plus the compares.  In 4 dimensions
// that is cheap and beats a shared-memory table (measured, round 1: config 2 0.740 -> 0.770 ms, config 3 0.551 ->
// 0.577 ms with the table: the shared-memory round trip sits on the node-to-node dependency chain).  In 10 dimensions
// the chains are a THIRD of everything the kernel executes (ncu, round 2, config 5 reduced: trace_core.cuh vsel 18.9 % +
// the axis line 13.4 % of all warp instructions, profiles/r02_c5s_dim10_ncu_summary.txt), so from NTR_SMEM_AXIS_MIN_DIM
// dimensions on the fixed-dimension kernels keep the three vectors in a per-thread column of shared memory instead
// (3*D floats per thread, column-major over the CTA: conflict-free for any mix of axes within a warp) and index it.
#ifndef NTR_SMEM_AXIS_MIN_DIM
#define NTR_SMEM_AXIS_MIN_DIM 9
#endif
#if defined(__CUDA_ARCH__)
#define NTR_AXIS_THREADS 128            // = kCtaThreads (kernels.cuh)
template <int DT> __device__ __forceinline__ float *axis_slab() {
    __shared__ float slab[3 * DimCap<DT>::value * NTR_AXIS_THREADS];
    return slab + threadIdx.x;
}
#define NTR_AXIS_IN_SMEM(DT) (DT >= NTR_SMEM_AXIS_MIN_DIM)
#define NTR_AXIS_SETUP(DT, D, o, dir, invdir)                                                              \
    float *axis_tab_ = nullptr;                                                                            \
    if (NTR_AXIS_IN_SMEM(DT)) {                                                                            \
        axis_tab_ = axis_slab<(NTR_AXIS_IN_SMEM(DT) ? DT : 1)>();                                          \
        _Pragma("unroll")                                                                                  \
        for (int i_ = 0; i_ < (DT > 0 ? DT : 1); ++i_) {                                                   \
            axis_tab_[i_ * NTR_AXIS_THREADS] = (o)[i_];                                                    \
            axis_tab_[(DT + i_) * NTR_AXIS_THREADS] = (dir)[i_];                                           \
            axis_tab_[(2 * DT + i_) * NTR_AXIS_THREADS] = (invdir)[i_];                                    \
        }                                                                                                  \
    }
#define NTR_AXIS_O(DT, o, axis) (NTR_AXIS_IN_SMEM(DT) ? axis_tab_[(axis) * NTR_AXIS_THREADS] : vsel<DT>(o, axis))
#define NTR_AXIS_DIR(DT, dir, axis) (NTR_AXIS_IN_SMEM(DT) ? axis_tab_[(DT + (axis)) * NTR_AXIS_THREADS] : vsel<DT>(dir, axis))
#define NTR_AXIS_INV(DT, invdir, axis) (NTR_AXIS_IN_SMEM(DT) ? axis_tab_[(2 * DT + (axis)) * NTR_AXIS_THREADS] : vsel<DT>(invdir, axis))
#else
#define NTR_AXIS_SETUP(DT, D, o, dir, invdir)
#define NTR_AXIS_O(DT, o, axis) vsel<DT>(o, axis)
#define NTR_AXIS_DIR(DT, dir, axis) vsel<DT>(dir, axis)
#define NTR_AXIS_INV(DT, invdir, axis) vsel<DT>(invdir, axis)
#endif

// ---- nearest-hit traversal ----------------------------------------------------------------------------
// kd_node_intersection::operator() (tracer.hpp:1179-1243) as an explicit stack machine.  Two frame
// kinds reproduce the recursion exactly: AFTER_NEAR (pending far child, split distance t, the caller's
// t_far, transparent-list size at entry) and AFTER_FAR (the near subtree hit beyond the split plane:
// the call returns true whatever the far subtree finds, and trims on a far hit, :1225-1230).
struct TravStack {
    uint32_t node[NTR_STACK_CAP];       // far child | AFTER_FAR marker
    float t[NTR_STACK_CAP];
    float t_far[NTR_STACK_CAP];
    unsigned char h_start[NTR_STACK_CAP];
};
#define NTR_FRAME_AFTER_FAR 0xFFFFFFFEu

template <int DT, int FLAGS>
NTR_HD bool trace_nearest(const SceneDev &s, const float *o, const float *dir, Skip skip, float t_near, float t_far,
                          HitRec &oh, GenState<DT> *g, Counters &cnt) {
    RaySlab<DT> rs;
    rs.init(s, dir);
    const float *invdir = rs.invdir;
    NTR_AXIS_SETUP(DT, NTR_D(DT, s), o, dir, invdir)
    TravStack st;
    int sp = 0;
    uint32_t node = s.root;
    MiniMailbox mm;
    if (FLAGS & NTR_F_GENERAL) { g->mb.clear(); } else { mm.clear(); }
    for (;;) {
        // ---- descend to a leaf (or fall off the tree) ----
        bool result = false;
        while (node != NTR_NULL_NODE) {
            const uint4 n = ldnode(s.nodes + node);
            if (n.x & NTR_LEAF_FLAG) {
#if NTR_CHUNKED_LEAVES
                if ((FLAGS & NTR_F_GENERAL) && n.z >= NTR_CHUNK_LEAF_MIN) result = leaf_general_chunked<DT, FLAGS>(s, n, o, dir, rs, skip, oh, *g, cnt);
                else
#endif
                if (FLAGS & NTR_F_GENERAL) result = leaf_general<DT, FLAGS>(s, n, o, dir, rs, skip, oh, *g, cnt);
                else result = leaf_opaque<DT, FLAGS>(s, n, o, dir, rs, skip, oh, mm, cnt);
                break;
            }
            if (FLAGS & NTR_F_COUNT) cnt.node_steps++;
            const int axis = (int)n.x;
            const float split = u2f(n.y);
            const float da = NTR_AXIS_DIR(DT, dir, axis), oa = NTR_AXIS_O(DT, o, axis);
            if (da != 0) {
                if (oa == split) { node = da > 0 ? n.w : n.z; continue; }
                const float t = (split - oa) * NTR_AXIS_INV(DT, invdir, axis);
                const uint32_t n_near = oa > split ? n.w : n.z;
                const uint32_t n_far = oa > split ? n.z : n.w;
                if (t < 0 || t > t_far) { node = n_near; continue; }
                if (t < t_near) { node = n_far; continue; }
                if (n_near != NTR_NULL_NODE) {
                    if (n_far == NTR_NULL_NODE) { node = n_near; t_far = t; continue; }   // `|| !n_far) return hit`
                    if (sp < NTR_STACK_CAP) {
                        st.node[sp] = n_far; st.t[sp] = t; st.t_far[sp] = t_far;
                        if (FLAGS & NTR_F_GENERAL) st.h_start[sp] = (unsigned char)g->th.n;
                        ++sp;
                    }
                    node = n_near;
                    t_far = t;
                    continue;
                }
                node = n_far;
                t_near = t;
                continue;
            }
            node = oa >= split ? n.w : n.z;
        }
        // ---- unwind ----
        for (;;) {
            if (sp == 0) return result;
            --sp;
            const uint32_t fnode = st.node[sp];
            if (fnode == NTR_FRAME_AFTER_FAR) {
                if (FLAGS & NTR_F_GENERAL) { if (result) g->th.trim(oh.dist, st.h_start[sp]); }
                result = true;
                continue;
            }
            const float t = st.t[sp];
            if (result && oh.dist <= t) continue;                   // tracer.hpp:1214
            node = fnode;
            t_near = t;
            t_far = st.t_far[sp];
            if (result) {                                           // tracer.hpp:1216-1231
                st.node[sp] = NTR_FRAME_AFTER_FAR;                  // h_start[sp] stays
                ++sp;
            }
            break;
        }
    }
}

// ---- occlusion (shadow) traversal ------------------------------------------------------------------------
// kd_leaf::occludes (tracer.hpp:1088-1124): any opaque hit nearer than the light blocks; transparent
// blockers are collected (no mailbox here).
template <int DT, int FLAGS>
NTR_HD bool leaf_occludes(const SceneDev &s, const uint4 node, const float *o, const float *dir, const RaySlab<DT> &rs,
                          float ldistance, Skip skip, HitList *hits, Counters &cnt) {
    const uint2 *items = s.leaf_items + node.y;
    const uint32_t size = node.z;
    for (uint32_t i = 0; i < size; ++i) {
        const uint2 it = lditem(items + i);
        const uint32_t item = it.x, off = it.y;
        const uint32_t kind = item >> 30;
        uint32_t meta = 0;
        float dist;
        int lane = -1;
        if (kind == NTR_REF_BATCH) {
            lane = skip.ref == item ? skip.lane : -1;
            dist = batch_test<DT, FLAGS>(s, off, o, dir, lane, ldistance, meta, cnt);
        } else {
            if (item == skip.ref) continue;
            if (kind == NTR_REF_SIMPLEX) {
                if (FLAGS & NTR_F_COUNT) cnt.simplex_tests++;
                dist = simplex_single<DT>(s, off, o, dir, ldistance, meta);
            } else if (FLAGS & NTR_F_GENERAL) {
                float P[DimCap<DT>::value], N[DimCap<DT>::value];
                uint32_t wmask;
                if (FLAGS & NTR_F_COUNT) cnt.solid_tests++;
                dist = solid_test<DT>(s, item & NTR_IDX_MASK, o, dir, ldistance, P, N, wmask, meta);
            } else {
                dist = 0;
            }
        }
        if (dist) {
            if (!(FLAGS & NTR_F_GENERAL) || (meta & NTR_META_OPAQUE)) return true;
            hits->add(dist, item, lane);
        }
    }
    return false;
}

// _occludes (tracer.hpp:1258-1307), including `if(t < ldistance) return false` (:1298): the far child is
// only entered when the split plane is farther away than the light.
template <int DT, int FLAGS>
NTR_HD bool trace_occludes(const SceneDev &s, const float *o, const float *dir, float ldistance, Skip skip,
                           float t_near, float t_far, HitList *hits, Counters &cnt) {
    RaySlab<DT> rs;
    rs.init(s, dir);
    const float *invdir = rs.invdir;
    NTR_AXIS_SETUP(DT, NTR_D(DT, s), o, dir, invdir)
    uint32_t st_node[NTR_STACK_CAP];
    float st_t[NTR_STACK_CAP], st_tfar[NTR_STACK_CAP];
    int sp = 0;
    uint32_t node = s.root;
    for (;;) {
        while (node != NTR_NULL_NODE) {
            const uint4 n = ldnode(s.nodes + node);
            if (n.x & NTR_LEAF_FLAG) {
                if (leaf_occludes<DT, FLAGS>(s, n, o, dir, rs, ldistance, skip, hits, cnt)) return true;
                break;
            }
            if (FLAGS & NTR_F_COUNT) cnt.node_steps++;
            const int axis = (int)n.x;
            const float split = u2f(n.y);
            const float da = NTR_AXIS_DIR(DT, dir, axis), oa = NTR_AXIS_O(DT, o, axis);
            if (da != 0) {
                if (oa == split) { node = da > 0 ? n.w : n.z; continue; }
                const float t = (split - oa) * NTR_AXIS_INV(DT, invdir, axis);
                const uint32_t n_near = oa > split ? n.w : n.z;
                const uint32_t n_far = oa > split ? n.z : n.w;
                if (t < 0 || t > t_far) { node = n_near; continue; }
                if (t < t_near) { node = n_far; continue; }
                if (n_near != NTR_NULL_NODE) {
                    if (n_far == NTR_NULL_NODE) { t_far = t; node = n_near; continue; }
                    if (sp < NTR_STACK_CAP) { st_node[sp] = n_far; st_t[sp] = t; st_tfar[sp] = t_far; ++sp; }
                    node = n_near;
                    t_far = t;
                    continue;
                }
                if (t < ldistance) break;           // near child null: falls to the same test (:1297-1298)
                t_near = t;
                node = n_far;
                continue;
            }
            node = oa >= split ? n.w : n.z;
        }
        // the (sub)call returned false: resume the innermost pending far child
        for (;;) {
            if (sp == 0) return false;
            --sp;
            if (st_t[sp] < ldistance) continue;     // `return false` of that frame
            node = st_node[sp];
            t_near = st_t[sp];
            t_far = st_tfar[sp];
            break;
        }
    }
}

// ---- shading ------------------------------------------------------------------------------------------
struct Mat { float c[3], spec[3], opacity, reflectivity, spec_int, spec_exp; };
NTR_HD Mat load_mat(const SceneDev &s, uint32_t meta) {
    const float *m = s.materials + (size_t)(meta & 0x7FFFFFFFu) * 12;
    const float4 a = ld4(m), b = ld4(m + 4), c = ld4(m + 8);
    Mat r;
    r.c[0] = a.x; r.c[1] = a.y; r.c[2] = a.z; r.spec[0] = a.w; r.spec[1] = b.x; r.spec[2] = b.y;
    r.opacity = b.z; r.reflectivity = b.w; r.spec_int = c.x; r.spec_exp = c.y;
    return r;
}

// composite_scene::light_reaches (tracer.hpp:1750-1766): false when blocked, else multiplies `filtered`
// by (1 - opacity) of every distinct transparent blocker.
template <int DT, int FLAGS>
NTR_HD bool light_reaches(const SceneDev &s, const float *o, const float *dir, float ldistance, Skip skip,
                          float *filtered, Counters &cnt) {
    HitList hits;
    if (FLAGS & NTR_F_GENERAL) hits.clear();
    cnt.shadow_rays++;
    if (trace_occludes<DT, FLAGS>(s, o, dir, ldistance, skip, 0.0f, FLT_MAX, &hits, cnt)) return false;
    if (FLAGS & NTR_F_GENERAL) {
        if (hits.dropped) cnt.truncated++;
        if (hits.n) {
            hits.sort_and_unique();
            for (int i = hits.n - 1; i >= 0; --i) {
                const Mat m = load_mat(s, target_meta<DT>(s, hits.ref[i], hits.lane[i]));
                const float f = 1 - m.opacity;
                filtered[0] *= f; filtered[1] *= f; filtered[2] *= f;
            }
        }
    }
    return true;
}

// append_specular (tracer.hpp:1701-1707), Blinn-Phong as written there (including `c *= a`).
template <int DT>
NTR_HD void append_specular(const SceneDev &s, float *spec, float &a, const Mat &m, const float *light_c,
                            const float *view, const float *normal, const float *light_dir) {
    const int D = NTR_D(DT, s);
    float h[DimCap<DT>::value];
    float sq = 0;
    NTR_UNROLL
    for (int i = 0; i < D; ++i) { h[i] = light_dir[i] - view[i]; sq += h[i] * h[i]; }
    const float len = sqrtf(sq);
    float dn = 0;
    NTR_UNROLL
    for (int i = 0; i < D; ++i) dn += normal[i] * (h[i] / len);
    const float base = powf(dn, m.spec_exp) * m.spec_int;
    const float k = base * (1 - a);
    NTR_UNROLL
    for (int c = 0; c < 3; ++c) spec[c] += m.spec[c] * light_c[c] * k;
    a += k;
    NTR_UNROLL
    for (int c = 0; c < 3; ++c) spec[c] *= a;
}

// point_light::strength (tracer.hpp:1686-1688): 1/dist^(D-1), evaluated in double like std::pow(float,size_t)
NTR_HD float light_strength(float dist, int D) {
    double p = 1.0, d = (double)dist;
    for (int i = 0; i < D - 1; ++i) p *= d;
    return (float)(1.0 / p);
}

// A deferred reflection bounce (tracer.hpp:1842-1851 linearised: the recursive colour enters the parent
// linearly, so the child ray carries the RGB weight c * reflectivity * (1 - spec_a) * parent weight).
template <int DT> struct Bounce {
    float o[DimCap<DT>::value], d[DimCap<DT>::value];
    float w[3];
    Skip skip;
    int depth;
};

// composite_scene::base_color (tracer.hpp:1768-1854) in three pieces, so that the per-lane version below (shade_hit) and
// the warp-synchronous one (trace_warp.cuh: shadow rays of a whole warp traced together) share every line of arithmetic:
//   light_prepare   geometry of one light at the hit: direction, distance, sine, strength; says whether the light
//                   contributes at all and whether a shadow ray decides it
//   light_apply     adds the light (after light_reaches filtered its colour) and its Blinn-Phong term, in light order
//   shade_finish    camera light, ambient + diffuse, the deferred reflection ray, accumulation into `acc`
template <int DT> struct LightSample {
    float lv[DimCap<DT>::value];
    float dist, sine, strength;
    float lc[3];
    bool is_point;
};
struct ShadeAcc { float light[3], spec[3], spec_a; };
enum : int { NTR_LIGHT_NONE = 0, NTR_LIGHT_DIRECT = 1, NTR_LIGHT_SHADOWED = 2 };

template <int DT>
NTR_HD int light_prepare(const SceneDev &s, int li, const float *P, const float *N, LightSample<DT> &ls) {
    const int D = NTR_D(DT, s);
    ls.is_point = li < s.n_point;
    const float *L = ls.is_point ? s.point_lights + (size_t)li * (D + 3) : s.global_lights + (size_t)(li - s.n_point) * (D + 3);
    ls.lc[0] = ldf(L + D); ls.lc[1] = ldf(L + D + 1); ls.lc[2] = ldf(L + D + 2);
    ls.dist = FLT_MAX; ls.sine = 0; ls.strength = 1.0f;
    if (ls.is_point) {
        float sq = 0;
    NTR_UNROLL
        for (int i = 0; i < D; ++i) { ls.lv[i] = P[i] - ldf(L + i); sq += ls.lv[i] * ls.lv[i]; }
        ls.dist = sqrtf(sq);
    NTR_UNROLL
        for (int i = 0; i < D; ++i) { ls.lv[i] /= ls.dist; ls.sine += N[i] * ls.lv[i]; }
    } else {
    NTR_UNROLL
        for (int i = 0; i < D; ++i) { ls.lv[i] = -ldf(L + i); ls.sine += N[i] * ls.lv[i]; }
    }
    if (!(ls.sine > 0)) return NTR_LIGHT_NONE;
    if (ls.is_point) ls.strength = light_strength(ls.dist, D);
    if (!s.shadows) return NTR_LIGHT_DIRECT;
    // LIGHT_THRESHOLD applies to point lights only, and drops the light entirely (tracer.hpp:1784-1803)
    if (ls.is_point && !(fmaxf(ls.lc[0], fmaxf(ls.lc[1], ls.lc[2])) * ls.strength * ls.sine > NTR_LIGHT_THRESHOLD)) return NTR_LIGHT_NONE;
    return NTR_LIGHT_SHADOWED;
}

// `filtered` = the light's colour as light_reaches left it (NTR_LIGHT_SHADOWED only)
template <int DT>
NTR_HD void light_apply(const SceneDev &s, int kind, const LightSample<DT> &ls, float *filtered, const Mat &m,
                        const float *view, const float *N, ShadeAcc &a) {
    if (kind == NTR_LIGHT_SHADOWED) {
        if (ls.is_point) { filtered[0] *= ls.strength; filtered[1] *= ls.strength; filtered[2] *= ls.strength; }
    NTR_UNROLL
        for (int c = 0; c < 3; ++c) a.light[c] += filtered[c] * ls.sine;
        if (m.spec_int != 0) append_specular<DT>(s, a.spec, a.spec_a, m, filtered, view, N, ls.lv);
    } else if (ls.is_point) {
    NTR_UNROLL
        for (int c = 0; c < 3; ++c) a.light[c] += ls.lc[c] * ls.strength * ls.sine;
    } else {
    NTR_UNROLL
        for (int c = 0; c < 3; ++c) a.light[c] += ls.lc[c] * ls.sine;
    }
}

// Returns true and fills `b` when a reflection ray follows.
template <int DT>
NTR_HD bool shade_finish(const SceneDev &s, const Mat &m, const float *view, const float *P, const float *N, Skip source,
                         int depth, const float *w, float *acc, ShadeAcc &a, Bounce<DT> &b, Counters &cnt) {
    const int D = NTR_D(DT, s);
    float sine = 0;
    NTR_UNROLL
    for (int i = 0; i < D; ++i) sine += view[i] * N[i];
    sine = -sine;
    if (s.camera_light && sine > 0) {
    NTR_UNROLL
        for (int c = 0; c < 3; ++c) a.light[c] += sine;
        if (m.spec_int != 0) {
            const float base = powf(sine, m.spec_exp) * m.spec_int;
            const float k = base * (1 - a.spec_a);
    NTR_UNROLL
            for (int c = 0; c < 3; ++c) a.spec[c] += m.spec[c] * k;
            a.spec_a += k;
    NTR_UNROLL
            for (int c = 0; c < 3; ++c) a.spec[c] *= a.spec_a;
        }
    }

    const bool reflect = m.reflectivity != 0 && depth < s.max_depth;
    const float keep = (reflect ? (1 - m.reflectivity) : 1.0f) * (1 - a.spec_a);
    NTR_UNROLL
    for (int c = 0; c < 3; ++c) {
        const float local = s.ambient[c] + m.c[c] * a.light[c];
        acc[c] += w[c] * (a.spec[c] + local * keep);
    }
    if (reflect) {
        const float k = m.reflectivity * (1 - a.spec_a);
    NTR_UNROLL
        for (int i = 0; i < D; ++i) { b.o[i] = P[i]; b.d[i] = view[i] - N[i] * (-2 * sine); }
    NTR_UNROLL
        for (int c = 0; c < 3; ++c) b.w[c] = w[c] * m.c[c] * k;
        b.skip = source;
        b.depth = depth + 1;
        cnt.reflection_rays++;
    }
    return reflect;
}

// base_color for one hit (P, N) of primitive (ref, lane), with the result multiplied by `w` and added to `acc`.
template <int DT, int FLAGS>
NTR_HD bool shade_hit(const SceneDev &s, const float *view, const float *P, const float *N, uint32_t ref, int lane,
                      int depth, const float *w, float *acc, Bounce<DT> &b, Counters &cnt) {
    const Mat m = load_mat(s, target_meta<DT>(s, ref, lane));
    const Skip source = {ref, lane};
    ShadeAcc a = {{0, 0, 0}, {0, 0, 0}, 0};
    cnt.shaded_hits++;
    // point lights first, then global lights (tracer.hpp:1776-1827), as ONE loop so that the shadow traversal
    // (light_reaches) is instantiated once
    const int n_lights = s.n_point + s.n_global;
    for (int li = 0; li < n_lights; ++li) {
        LightSample<DT> ls;
        const int kind = light_prepare<DT>(s, li, P, N, ls);
        if (kind == NTR_LIGHT_NONE) continue;
        float filtered[3] = {ls.lc[0], ls.lc[1], ls.lc[2]};
        if (kind == NTR_LIGHT_SHADOWED && !light_reaches<DT, FLAGS>(s, P, ls.lv, ls.dist, source, filtered, cnt)) continue;
        light_apply<DT>(s, kind, ls, filtered, m, view, N, a);
    }
    return shade_finish<DT>(s, m, view, P, N, source, depth, w, acc, a, b, cnt);
}

// composite_scene::aabb_distance (tracer.hpp:1892-1918)
template <int DT> NTR_HD float aabb_distance(const SceneDev &s, const float *o, const float *dir) {
    const int D = NTR_D(DT, s);
    for (int i = 0; i < D; ++i) {
        const float di = vsel<DT>(dir, i);
        if (di != 0) {
            const float oi = vsel<DT>(o, i);
            const float plane = di > 0 ? vsel<DT>(s.bmin, i) : vsel<DT>(s.bmax, i);
            float dist = (plane - oi) / di;
            int skip = i;
            if (dist < 0) { dist = 0; skip = -1; }
            bool miss = false;
    NTR_UNROLL
            for (int j = 0; j < D; ++j) {
                if (j != skip) {
                    const float v = dir[j] * dist + o[j];
                    if (v >= s.bmax[j] || v <= s.bmin[j]) miss = true;
                }
            }
            if (!miss) return dist;
        }
    }
    return -1;
}

// hit geometry for list entries and for the opaque hit of the fast variant
template <int DT, int FLAGS>
NTR_HD void hit_geometry(const SceneDev &s, uint32_t ref, int lane, float dist, const float *o, const float *dir,
                         float *P, float *N) {
    const uint32_t kind = ref >> 30, idx = ref & NTR_IDX_MASK;
    if (kind == NTR_REF_SOLID) {
        if (FLAGS & NTR_F_GENERAL) {
            uint32_t wmask, meta;
            solid_test<DT>(s, idx, o, dir, FLT_MAX, P, N, wmask, meta);
        }
        return;
    }
    simplex_normal<DT>(s, kind == NTR_REF_BATCH ? idx + (uint32_t)lane : idx, o, dir, dist, P, N);
}

// composite_scene::ray_color (tracer.hpp:1856-1883), linearised: the transparent layers (sorted near to
// far) and the opaque hit / background each contribute base_color * op_i * prod_{j<i}(1 - op_j).
// EMIT(const Bounce<DT>&) receives the deferred reflection rays.  normal_out (D floats, left alone on a miss) receives
// the normal that shades the opaque hit.
template <int DT, int FLAGS, typename EMIT>
NTR_HD void ray_color(const SceneDev &s, bool enabled, const float *o, const float *dir, int depth, Skip source,
                      const float *weight, float *acc, EMIT &emit, Counters &cnt, HitRec *primary_out,
                      MailboxStore *ms = nullptr, float *normal_out = nullptr) {
    const int D = NTR_D(DT, s);
    GenState<DT> g;
    g.mb.big = (ms && ms->col) ? ms : nullptr;
    HitRec oh;
    oh.dist = FLT_MAX; oh.ref = NTR_NONE_REF; oh.lane = -1;
    if (FLAGS & NTR_F_GENERAL) {
        g.th.clear();
    NTR_UNROLL
        for (int i = 0; i < D; ++i) { g.hitP[i] = 0; g.hitN[i] = 0; }
    }
    const float t0 = enabled ? aabb_distance<DT>(s, o, dir) : -1.0f;
    const bool hit = t0 >= 0 && trace_nearest<DT, FLAGS>(s, o, dir, source, t0, FLT_MAX, oh, &g, cnt);
    if (!enabled) return;
    if (primary_out) { *primary_out = oh; if (!hit) { primary_out->ref = NTR_NONE_REF; primary_out->dist = 0; } }

    float w[3] = {weight[0], weight[1], weight[2]};
    float P[DimCap<DT>::value], N[DimCap<DT>::value];
    Bounce<DT> b;
    // layers near -> far: the surviving transparent hits (sorted, unique), then the opaque hit.  One loop, one
    // shade_hit call site (keeps a single copy of the shading + shadow-traversal code in the kernel).
    int n_layers = 0;
    if (FLAGS & NTR_F_GENERAL) {
        if (g.th.dropped) cnt.truncated++;          // the list outgrew NTR_THITS_CAP: reported, ntr_counters.truncated_hit_lists
        if (g.th.n) g.th.sort_and_unique();
        n_layers = g.th.n;
    }
    const int n_total = n_layers + (hit ? 1 : 0);
    for (int i = 0; i < n_total; ++i) {
        uint32_t ref;
        int lane;
        float wl[3];
        if (i < n_layers) {
            ref = g.th.ref[i];
            lane = g.th.lane[i];
            const float op = load_mat(s, target_meta<DT>(s, ref, lane)).opacity;
            hit_geometry<DT, FLAGS>(s, ref, lane, g.th.dist[i], o, dir, P, N);
            wl[0] = w[0] * op; wl[1] = w[1] * op; wl[2] = w[2] * op;
            w[0] *= 1 - op; w[1] *= 1 - op; w[2] *= 1 - op;
        } else {
            ref = oh.ref;
            lane = oh.lane;
            wl[0] = w[0]; wl[1] = w[1]; wl[2] = w[2];
            if (FLAGS & NTR_F_GENERAL) {
    NTR_UNROLL
                for (int k = 0; k < D; ++k) { P[k] = g.hitP[k]; N[k] = g.hitN[k]; }      // as the reference left it (Q12)
            } else {
                hit_geometry<DT, FLAGS>(s, ref, lane, oh.dist, o, dir, P, N);
            }
            if (normal_out) {
    NTR_UNROLL
                for (int k = 0; k < D; ++k) normal_out[k] = N[k];
            }
        }
        if (shade_hit<DT, FLAGS>(s, dir, P, N, ref, lane, depth, wl, acc, b, cnt)) emit(b);
    }
    if (!hit) {
        const float I = vsel<DT>(dir, s.bg_axis);       // tracer.hpp:1866-1867
    NTR_UNROLL
        for (int c = 0; c < 3; ++c) {
            const float bg = I >= 0 ? s.bg1[c] * I + s.bg2[c] * (1 - I) : s.bg3[c] * -I + s.bg2[c] * (1 + I);
            acc[c] += w[c] * bg;
        }
    }
}

// flat_origin_ray_source::operator() (tracer.hpp:71-75): integer pixel coordinates, no half-pixel offset
template <int DT>
NTR_HD void primary_ray_of(const SceneDev &s, const CameraDev &cam, float fovI, float half_w, float half_h, int x, int y,
                           float *o, float *dir) {
    const int D = NTR_D(DT, s);
    const float fx = fovI * ((float)x - half_w), fy = fovI * ((float)y - half_h);
    float sq = 0;
    NTR_UNROLL
    for (int i = 0; i < D; ++i) {
        o[i] = cam.origin[i];
        dir[i] = cam.fwd[i] + cam.right[i] * fx - cam.up[i] * fy;
        sq += dir[i] * dir[i];
    }
    const float len = sqrtf(sq);
    NTR_UNROLL
    for (int i = 0; i < D; ++i) dir[i] /= len;
}

// ---- projections (ntr_scene_set_projection; no counterpart in the reference) ----------------------------------------
// The parameter of projection `kind` for a view of half width half_w: k = h / half_w (orthographic: scene units per pixel)
// or a = alpha / (2 * half_w) (equirectangular: radians per pixel), in float like fovI.  At factor s the view's half_w is
// s times the plain one, so k and a scale by 1/s exactly when s is a power of two.
NTR_HD float projection_k(int kind, float param, float half_w) {
    return kind == NTR_PROJ_ORTHOGRAPHIC ? param / half_w : param / (2.0f * half_w);
}
// pixel (x, y) of a view under an orthographic (kind 1) or equirectangular (kind 2) projection with parameter k
template <int DT>
NTR_HD void projected_ray_of(const SceneDev &s, const CameraDev &cam, int kind, float k, float half_w, float half_h, int x, int y,
                             float *o, float *dir) {
    const int D = NTR_D(DT, s);
    const float u = k * ((float)x - half_w), v = k * ((float)y - half_h);
    float sq = 0;
    if (kind == NTR_PROJ_ORTHOGRAPHIC) {
    NTR_UNROLL
        for (int i = 0; i < D; ++i) {
            o[i] = cam.origin[i] + cam.right[i] * u - cam.up[i] * v;
            dir[i] = cam.fwd[i];
            sq += dir[i] * dir[i];
        }
    } else {
        const float st = sinf(u), ct = cosf(u), sp = sinf(v), cp = cosf(v);
    NTR_UNROLL
        for (int i = 0; i < D; ++i) {
            o[i] = cam.origin[i];
            dir[i] = cp * (st * cam.right[i] + ct * cam.fwd[i]) - sp * cam.up[i];
            sq += dir[i] * dir[i];
        }
    }
    const float len = sqrtf(sq);
    NTR_UNROLL
    for (int i = 0; i < D; ++i) dir[i] /= len;
}
// The primary ray of pixel (x, y): PROJ (the NTR_F_PROJ builds and camera_rays_kernel) switches on the projection kind at run
// time; without it the code is the pinhole's alone.
template <int DT, bool PROJ>
NTR_HD void primary_ray_at(const SceneDev &s, const CameraDev &cam, int proj, float proj_k, float fovI, float half_w, float half_h,
                           int x, int y, float *o, float *dir) {
    if constexpr (PROJ) {
        if (proj != NTR_PROJ_PERSPECTIVE) {
            projected_ray_of<DT>(s, cam, proj, proj_k, half_w, half_h, x, y, o, dir);
            return;
        }
    }
    primary_ray_of<DT>(s, cam, fovI, half_w, half_h, x, y, o, dir);
}
template <int DT, bool PROJ = false>
NTR_HD void primary_ray(const SceneDev &s, const CameraDev &cam, const FrameDev &f, int x, int y, float *o, float *dir) {
    primary_ray_at<DT, PROJ>(s, cam, f.proj, f.proj_k, f.fovI, f.half_w, f.half_h, x, y, o, dir);
}

// box_scene::calculate_color (tracer.hpp:101-114) with hypercube_intersects (:126-152) inlined:
// the unit hypercube at the origin, fixed shading, gradient background.
// normal_out (D floats, left alone on a miss): the axis vector of the face that was hit
template <int DT>
NTR_HD void box_color(const SceneDev &s, const float *o, const float *dir, float *rgb, HitRec *primary_out,
                      float *normal_out = nullptr) {
    const int D = NTR_D(DT, s);
    for (int i = 0; i < D; ++i) {
        const float di = vsel<DT>(dir, i);
        if (di != 0) {
            const float face = di < 0 ? 1.0f : -1.0f;
            const float dist = (face - vsel<DT>(o, i)) / di;
            if (dist > 0) {
                bool miss = false;
    NTR_UNROLL
                for (int j = 0; j < D; ++j) {
                    if (j != i) { if (fabsf(dir[j] * dist + o[j]) > (1 + NTR_FUZZ)) miss = true; }
                }
                if (!miss) {
                    const float sine = di * face;           // dot(view.direction, axis(i, face))
                    const float k = sine <= 0 ? -sine : 0.0f;
                    rgb[0] = k * 1.0f; rgb[1] = k * 0.5f; rgb[2] = k * 0.5f;
                    if (primary_out) { primary_out->dist = dist; primary_out->ref = 0; primary_out->lane = -1; }
                    if (normal_out) for (int j = 0; j < D; ++j) normal_out[j] = j == i ? face : 0.0f;
                    return;
                }
            }
        }
    }
    const float I = dir[0];
    if (I > 0) { rgb[0] = I; rgb[1] = I; rgb[2] = I; }
    else { rgb[0] = 0; rgb[1] = -I; rgb[2] = -I; }
    if (primary_out) { primary_out->dist = 0; primary_out->ref = NTR_NONE_REF; primary_out->lane = -1; }
}

// ---- supersampling (ntr_scene_set_supersampling; no counterpart in the reference) ----------------------------------
// Output pixel (x, y) of a frame with factor ss = f.ss > 1 is the box-filtered mean of pixels (ss*x + i, ss*y + j) of the
// ss-times-larger view that f describes, summed j-major, i-minor.  Every sample is traced from zero exactly as the big
// view's pixel, with weight 1/ss^2 from the start, so its bounces (emitted to the next pass with that weight) need nothing
// special.  Scaling by a power of two is exact and no decision of the per-ray code reads the weight: for ss in {2, 4, 8}
// the per-sample colours are the big view's times 1/ss^2 and their sum is the big view's float32 sequential box sum times
// 1/ss^2, bit for bit.  The sum is added without contraction so that it cannot fuse with the last product of a sample.
NTR_HD float add_rn(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fadd_rn(a, b);
#else
    return a + b;
#endif
}
NTR_HD float mul_rn(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fmul_rn(a, b);
#else
    return a * b;
#endif
}

// colour of output pixel (x, y) of a supersampled frame into sum[3]; samples go to the (per-lane) ray_color.
// EXACT1 (the primary pass of a batch of views, NTR_F_VIEWS, which runs factor 1 through here as well): at factor 1 the one
// sample's colour is stored as it is, so that the pixel has the bits of the plain primary path -- 0.0f + c would turn a
// negative zero into +0 (box_color stores -0 where the direction's gradient axis is +0; tests/test_views.py)
//
// aov (NTR_F_AOV): receives the hit of the pixel's plain (factor-1) primary ray.  For ss in {1, 2, 4, 8} that ray is sample
// (0, 0) bit for bit -- fovI / ss and ss * x - ss * half_w scale exactly by a power of two (tests/test_aovs.py) -- so its hit
// is taken from that sample's ray_color.  Any other factor traces the plain ray once more (plain_primary_hit).
template <int DT> struct PrimaryAov {
    HitRec hit;
    float n[DimCap<DT>::value];     // the normal that shades the hit; zeros on a miss
};
template <int DT, int FLAGS, bool PROJ = false>
NTR_HD void plain_primary_hit(const SceneDev &s, const CameraDev &cam, const FrameDev &f, int x, int y, PrimaryAov<DT> &a,
                              MailboxStore *ms);

// PROJ: the NTR_F_PROJ builds (primary_ray_at)
template <int DT, int FLAGS, typename EMIT, bool EXACT1 = false, bool PROJ = false>
NTR_HD void ss_pixel_color(const SceneDev &s, const CameraDev &cam, const FrameDev &f, int x, int y, float *sum,
                           EMIT &emit, Counters &cnt, MailboxStore *ms, PrimaryAov<DT> *aov = nullptr) {
    constexpr int CAP = DimCap<DT>::value;
    const int ss = f.ss;
    const bool pow2 = (ss & (ss - 1)) == 0;
    if (aov) {
        aov->hit.dist = 0; aov->hit.ref = NTR_NONE_REF; aov->hit.lane = -1;
        for (int i = 0; i < CAP; ++i) aov->n[i] = 0.0f;
    }
    const float wt = 1.0f / (float)(ss * ss);
    const float w[3] = {wt, wt, wt};
    const Skip none = {NTR_NONE_REF, 0};
    sum[0] = 0.0f; sum[1] = 0.0f; sum[2] = 0.0f;
    for (int k = 0; k < ss * ss; ++k) {
        const int j = k / ss, i = k - j * ss;
        float o[CAP], dir[CAP];
        float c[3] = {0.0f, 0.0f, 0.0f};
        primary_ray<DT, PROJ>(s, cam, f, ss * x + i, ss * y + j, o, dir);
        const bool capture = aov && pow2 && k == 0;
        if (s.kind == NTR_SCENE_BOX) {
            box_color<DT>(s, o, dir, c, capture ? &aov->hit : nullptr, capture ? aov->n : nullptr);   // assigns the colour: weight it here
            c[0] = mul_rn(c[0], wt); c[1] = mul_rn(c[1], wt); c[2] = mul_rn(c[2], wt);
        } else {
            ray_color<DT, FLAGS>(s, true, o, dir, 0, none, w, c, emit, cnt, capture ? &aov->hit : nullptr, ms,
                                 capture ? aov->n : nullptr);
        }
        if (EXACT1 && ss == 1) { sum[0] = c[0]; sum[1] = c[1]; sum[2] = c[2]; }
        else { sum[0] = add_rn(sum[0], c[0]); sum[1] = add_rn(sum[1], c[1]); sum[2] = add_rn(sum[2], c[2]); }
    }
    if (aov && !pow2) plain_primary_hit<DT, FLAGS, PROJ>(s, cam, f, x, y, *aov, ms);
}

// The hit of output pixel (x, y)'s plain primary ray, with the nearest-hit traversal of ray_color only: no shading, no
// bounces, no counters.  a must hold ray_color's miss state (ss_pixel_color clears it).
template <int DT, int FLAGS, bool PROJ>
NTR_HD void plain_primary_hit(const SceneDev &s, const CameraDev &cam, const FrameDev &f, int x, int y, PrimaryAov<DT> &a,
                              MailboxStore *ms) {
    constexpr int CAP = DimCap<DT>::value;
    constexpr int TF = FLAGS & ~NTR_F_COUNT;
    const int D = NTR_D(DT, s);
    float o[CAP], dir[CAP];
    primary_ray_at<DT, PROJ>(s, cam, f.proj, f.aov_proj_k, f.aov_fovI, f.aov_half_w, f.aov_half_h, x, y, o, dir);
    if (s.kind == NTR_SCENE_BOX) {
        float c[3];
        box_color<DT>(s, o, dir, c, &a.hit, a.n);
        return;
    }
    GenState<DT> g;
    g.mb.big = (ms && ms->col) ? ms : nullptr;
    HitRec oh;
    oh.dist = FLT_MAX; oh.ref = NTR_NONE_REF; oh.lane = -1;
    if (TF & NTR_F_GENERAL) {
        g.th.clear();
    NTR_UNROLL
        for (int i = 0; i < D; ++i) { g.hitP[i] = 0; g.hitN[i] = 0; }
    }
    Counters none;
    const Skip source = {NTR_NONE_REF, 0};
    const float t0 = aabb_distance<DT>(s, o, dir);
    if (!(t0 >= 0 && trace_nearest<DT, TF>(s, o, dir, source, t0, FLT_MAX, oh, &g, none))) return;
    a.hit = oh;
    if (TF & NTR_F_GENERAL) {
    NTR_UNROLL
        for (int k = 0; k < D; ++k) a.n[k] = g.hitN[k];
    } else {
        float P[CAP];
        hit_geometry<DT, TF>(s, oh.ref, oh.lane, oh.dist, o, dir, P, a.n);
    }
}

// ---- caller-given primary rays (ntr_render_rays; no counterpart in the reference) -------------------------------------
// The colour of primary ray (o, dir) into rgb[3], exactly as the plain primary pass colours a camera ray: box_color, or
// ray_color at depth 0 with no source and weight 1 into a zero accumulator.  The direction is used as given.
// aov (optional): receives the ray's opaque hit and the normal that shades it (ray_color's miss state and zeros on a miss).
template <int DT, int FLAGS, typename EMIT>
NTR_HD void given_ray_color(const SceneDev &s, const float *o, const float *dir, float *rgb, EMIT &emit, Counters &cnt,
                            MailboxStore *ms, PrimaryAov<DT> *aov) {
    if (aov) {
        aov->hit.dist = 0; aov->hit.ref = NTR_NONE_REF; aov->hit.lane = -1;
        for (int i = 0; i < DimCap<DT>::value; ++i) aov->n[i] = 0.0f;
    }
    rgb[0] = 0.0f; rgb[1] = 0.0f; rgb[2] = 0.0f;
    if (s.kind == NTR_SCENE_BOX) {
        box_color<DT>(s, o, dir, rgb, aov ? &aov->hit : nullptr, aov ? aov->n : nullptr);
        return;
    }
    const float one[3] = {1.0f, 1.0f, 1.0f};
    const Skip none = {NTR_NONE_REF, 0};
    ray_color<DT, FLAGS>(s, true, o, dir, 0, none, one, rgb, emit, cnt, aov ? &aov->hit : nullptr, ms, aov ? aov->n : nullptr);
}

// ---- adaptive supersampling (ntr_scene_set_supersampling_threshold) -------------------------------------------------
// Pixel (x, y) is refined -- traced again with ss_pixel_color -- iff, in some channel, the plain 1-spp colours of its
// corner set {(x, y), (x+1, y), (x, y+1), (x+1, y+1)} intersected with the view span more than the threshold.
//
// Accumulator slots of one launch: first the npix = win_w * out_rows pixels it owns, slot = out_row * win_w + x (out_row:
// the window row, or the row of the compacted strip of a sharded render); then the halo, the corner pixels the mask
// needs that the launch does not own, which it traces itself at factor 1 (no exchange between devices):
//   npix + r                                 pixel (win_w, row of output row r): the column right of the window
//   npix + out_rows + k * (win_w + 1) + x    pixel (x, row below the k-th owned tile row), when that row is not owned
// Slots whose pixel lies outside the view, or whose row is not a real owned row, are never traced or read.
NTR_HD int owned_tile_rows(const FrameDev &f) {
    return f.tile_row_first < f.tiles_y ? (f.tiles_y - f.tile_row_first + f.tile_row_step - 1) / f.tile_row_step : 0;
}
NTR_HD uint32_t halo_slots(const FrameDev &f) {
    return (uint32_t)f.out_rows + (uint32_t)owned_tile_rows(f) * (uint32_t)(f.win_w + 1);
}
// window row wy -> its output row, if this launch owns it
NTR_HD bool owned_row(const FrameDev &f, int wy, int *out_row) {
    if (wy < 0 || wy >= f.win_h) return false;
    const int ty = wy / NTR_TILE;
    if (ty < f.tile_row_first || (ty - f.tile_row_first) % f.tile_row_step != 0) return false;
    *out_row = f.compact ? (ty - f.tile_row_first) / f.tile_row_step * NTR_TILE + wy % NTR_TILE : wy;
    return true;
}
// output row -> window row (the inverse of owned_row; the row may lie past the window in the last tile of a strip)
NTR_HD int window_row(const FrameDev &f, int out_row) {
    return f.compact ? (f.tile_row_first + out_row / NTR_TILE * f.tile_row_step) * NTR_TILE + out_row % NTR_TILE : out_row;
}
// halo slot npix + h -> window pixel (wx, wy); false when the slot holds no pixel of this frame
NTR_HD bool halo_pixel(const FrameDev &f, uint32_t h, int *wx, int *wy) {
    const int vw = f.width / f.ss, vh = f.height / f.ss;
    int r = 0;
    if (h < (uint32_t)f.out_rows) {
        *wx = f.win_w;
        *wy = window_row(f, (int)h);
        return f.x0 + f.win_w < vw && owned_row(f, *wy, &r);
    }
    h -= (uint32_t)f.out_rows;
    const int k = (int)(h / (uint32_t)(f.win_w + 1));
    *wx = (int)(h % (uint32_t)(f.win_w + 1));
    const int ty = f.tile_row_first + k * f.tile_row_step;
    *wy = (ty + 1) * NTR_TILE < f.win_h ? (ty + 1) * NTR_TILE : f.win_h;
    return k < owned_tile_rows(f) && !owned_row(f, *wy, &r) && f.y0 + *wy < vh && f.x0 + *wx < vw;
}
// slot of corner pixel (wx, wy) of an owned pixel, or -1 when it lies outside the view
NTR_HD long long corner_slot(const FrameDev &f, int wx, int wy) {
    const int vw = f.width / f.ss, vh = f.height / f.ss;
    if (f.x0 + wx >= vw || f.y0 + wy >= vh) return -1;
    const long long npix = (long long)f.win_w * f.out_rows;
    int r = 0;
    if (owned_row(f, wy, &r)) return wx < f.win_w ? (long long)r * f.win_w + wx : npix + r;
    // the row above is owned: wy is the halo row below the k-th owned tile row
    const int k = ((wy - 1) / NTR_TILE - f.tile_row_first) / f.tile_row_step;
    return npix + f.out_rows + (long long)k * (f.win_w + 1) + wx;
}
// The refine rule for owned pixel (wx, wy) over the plain colours in accum (3 floats per slot): f describes the plain
// frame (factor 1), t >= 0 is the threshold.
NTR_HD bool refine_pixel(const FrameDev &f, const float *accum, int wx, int wy, float t) {
    float lo[3], hi[3];
    for (int c = 0; c < 4; ++c) {
        const long long slot = corner_slot(f, wx + (c & 1), wy + (c >> 1));
        if (slot < 0) continue;                     // (wx, wy) itself is always in the view
        for (int k = 0; k < 3; ++k) {
            const float v = accum[slot * 3 + k];
            lo[k] = c ? fminf(lo[k], v) : v;
            hi[k] = c ? fmaxf(hi[k], v) : v;
        }
    }
    return hi[0] - lo[0] > t || hi[1] - lo[1] > t || hi[2] - lo[2] > t;
}

// ---- pixel packing ------------------------------------------------------------------------------------
// process_pixel::operator() (reference src/render.cpp:421-462): channel = clamp(f_r*r+f_g*g+f_b*b+f_c,0,1);
// integer channels lround(v * double(2^bits-1)), float channels raw IEEE bits; bits appended MSB-first into
// a 128-bit big-endian accumulator.  out[0] holds the 4 most significant bytes (big-endian word order):
// byte j of the pixel = (out[j/4] >> (8*(3 - j%4))) & 0xff.
NTR_HD void pack_pixel(const FormatDev &f, const float *rgb, uint32_t out[4]) {
    unsigned long long hi = 0, lo = 0;
    int off = 0;
    for (int ci = 0; ci < f.n_channels; ++ci) {
        // ch.f_r*r + ch.f_g*g + ch.f_b*b + f_c (render.cpp:427), left to right and without FMA contraction: the
        // packed bytes are integer work and must not depend on how the compiler fuses this expression
#if defined(__CUDA_ARCH__)
        float v = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(f.f_r[ci], rgb[0]), __fmul_rn(f.f_g[ci], rgb[1])),
                                      __fmul_rn(f.f_b[ci], rgb[2])), f.f_c[ci]);
#else
        float v = f.f_r[ci] * rgb[0] + f.f_g[ci] * rgb[1] + f.f_b[ci] * rgb[2] + f.f_c[ci];
#endif
        v = fminf(fmaxf(v, 0.0f), 1.0f);
        const int bits = f.bits[ci];
        unsigned long long ival;
        if (f.tfloat[ci]) ival = f2u(v);
        else {
            // std::lround(val * double(0xffffffffu >> (32 - bit_size))), render.cpp:439
            ival = (unsigned long long)llround((double)v * (double)(0xffffffffu >> (32 - bits)));
        }
        const int o = off >> 6, rm = off & 63;
        const int sh = 64 - rm - bits;
        const unsigned long long part = sh >= 0 ? ival << sh : ival >> -sh;
        if (o == 0) hi |= part; else lo |= part;
        if (rm + bits > 64) lo = ival << (128 - rm - bits);
        off += bits;
    }
    out[0] = (uint32_t)(hi >> 32); out[1] = (uint32_t)hi; out[2] = (uint32_t)(lo >> 32); out[3] = (uint32_t)lo;
}

}  // namespace ntr
