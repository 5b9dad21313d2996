// rt_scene.cuh — device-resident scene layout and the closest-hit scan (HittableList::hit,
// /root/reference/src/shapes/mod.rs:56-69) of the B200 render path.
//
// Layout in HBM (built once by rtiow_scene_upload, read-only afterwards):
//   table    float [np/4+1][4][4]  filter table: one 64-byte record per 4 "small" spheres,
//                            [cx0..3][cy0..3][cz0..3][K0..3], K = |c|^2 - r^2 + R^2 lowered by the filter slack; list
//                            order, padded to whole 32-sphere words with never-hit entries (+1 record for the
//                            pipeline's look-ahead); staged into shared memory by each CTA and streamed as broadcast
//                            LDS.128 (4 spheres per load)
//   small    float4 [np]     (cx, cy, cz, r) exact f32 copy for the precise test of candidates
//   small_idx int   [np]     position in `small` -> index in the reference's list (-1 = padding)
//   big      double4 [nb]    (cx, cy, cz, r) spheres whose radius makes |oc|^2 - r^2 cancel in f32
//                            (the r=1000 ground, main.rs:64); tested in f64, 1 of ~530 tests
//   big_idx  int    [nb]
//   sph      float4 / double4 [n]  (cx,cy,cz,r) in list order, for HitRecord::new
//   mat      float4 / double4 [n]  (albedo r,g,b, fuzz|ir) resolved per sphere; kind uint8 [n]
#pragma once
#include "rt_device.cuh"
#include "rt_umma.cuh"

namespace rt {

struct SceneDev {
    const float* table;     // filter table, RT_TABLE_FLOATS(np) floats
    const float4* small;
    const int* small_idx;
    int np;                 // small spheres incl. padding: a multiple of 32
    int n_rec;              // 4-sphere records that hold real small spheres: ceil(ns / 4) <= np / 4
    float filter_R2;        // R^2: squared radius of the sphere around the coordinate origin that bounds every small sphere
    float filter_sigma;     // 16 u max|r|: per unit of |origin|_1, how far outside the R-sphere the filter's line point is put
    const double4* big;
    const int* big_idx;
    int nb;
    const float4* bigf;     // the same spheres for the f32 fast path: 3 float4 each: (c_hi, r), (c_lo, K_hi), (K_lo, |c|_1, 0, 0), K = |c|^2 - r^2
    const float4* sph;
    const double4* sphd;
    const float4* mat;
    const double4* matd;
    const uint8_t* kind;
    int n;
    // tensor-core filter (rt_umma.cuh, rt_umma_scan.cuh): the small spheres' feature rows, fp16 hi/lo, in the canonical
    // K-major layout tcgen05.mma reads from shared memory; u_npad = 0 when the scene does not qualify (too large for
    // shared memory, or so spread out that the fp16 split's slack would swamp the spheres)
    const unsigned char* u_bimg;   // [2][u_npad * 32] bytes: hi block, lo block
    int u_npad;                    // small spheres padded to a whole number of MMA chunks (never-pass entries)
    umma::FeatScale u_sc;
};

#define RT_FULL 0xffffffffu
// Conservative slack of the f32 filter, in units of (|c|^2 + r^2 + R^2): 96 * 2^-24.  The filter's rounding
// error is bounded by ~48 u (|c|^2 + R^2) + 4 u r^2 (u = 2^-24; derivation in DESIGN.md), so with this
// slack every sphere the precise test can accept passes the filter.  It is folded into K at upload: no cost
// inside the loop.
#define RT_FILTER_SLACK 5.7220458984375e-06f
#define RT_CAND_CAP 16           // candidate slots per lane per segment (uint16 positions)
#define RT_SEG_WORDS 32          // 32 words x 32 spheres per segment between drains

struct HitF {           // closest hit so far; t in units of the normalised direction
    float t;
    int idx;            // index in the reference's list, -1 = none
    int code;           // where the winner lives: >= 0 position in `small`, <= -2 : -2 - position in `big`, -1 none
};
#define RT_SELF_NONE (-1)

// Precise test of one candidate (sphere.rs:16-34 via sphere_roots), index-aware acceptance.
// The reference scans in list order and accepts root <= closest_so_far, so among equal roots the
// LARGEST index wins (sphere.rs:29,31; mod.rs:61-66); `t < best || (t == best && idx > best_idx)`
// gives the same winner for any processing order.
template <typename T, bool kSeededSqrt = false>
__device__ __forceinline__ void candidate(V3<T> o, V3<T> dhat, T inv_a, T t_min, V3<T> c, T r, int idx, T* t_best, int* i_best)
{
    T t;
    // t_max = +inf: a root beyond the current closest is rejected by the comparison below, exactly
    // as sphere.rs:29-33 rejects it (its far root is farther still)
    if (!sphere_roots<T, kSeededSqrt>(c - o, dhat, inv_a, r * r, t_min, (T)__int_as_float(0x7f800000), &t)) return;
    if (t < *t_best || (t == *t_best && idx > *i_best)) { *t_best = t; *i_best = idx; }
}

// The sphere a ray STARTS on (the one it just scattered from).  In f64 the reference's origin is within
// ~1e-15 of that surface, so its near-zero root never reaches t_min = 1e-4 (main.rs:44); an f32 origin
// is ~1e-6 off, which t_min * |dir| does not cover when the scattered direction is short
// (Lambertian normal + unit vector, materials.rs:23).  For that one sphere the origin is therefore
// taken ON the surface (centre + self_n * |r|, self_n = unit(p - centre)): the roots are exactly
// {0, 2 tca}, the zero root is dropped as sphere.rs:29 drops it, and only 2 tca is offered.
template <typename T>
__device__ __forceinline__ void candidate_self(V3<T> dhat, T inv_a, T t_min, V3<T> self_n, T r, int idx, T* t_best, int* i_best)
{
    const T t = T(-2) * abs_t(r) * dot(self_n, dhat) * inv_a;      // oc = -|r| self_n ; t = 2 (oc . dhat) / a
    if (!(t >= t_min)) return;
    if (t < *t_best || (t == *t_best && idx > *i_best)) { *t_best = t; *i_best = idx; }
}

// The f32 scan over the filter table (shared memory, or global when the scene does not fit).
//
//   Filter, all spheres, branch-free, packed f32x2 over sphere pairs: 7 FFMA2 per 2 tests, nothing else on the FP32 pipe.
//   sphere.rs:18-25 is oc = o - c; half_b = oc.d; c = |oc|^2 - r^2; disc = half_b^2 - a c.  The discriminant belongs to
//   the ray's LINE, so any point p of the line may stand in for the origin; expanded around the coordinate origin, with
//   a unit direction,
//       hb = c.d - p.d ;   C = (|c|^2 - r^2 + |p|^2) - 2 c.p ;   disc' = hb^2 - C .
//   Per-ray and per-sphere parts separate except for |p|^2 — so p is chosen ON THE SPHERE |p| = R around the coordinate
//   origin (R = SceneDev::filter_R2^(1/2), a bound of all small spheres, fixed at upload): then |p|^2 = R^2 is a constant
//   of the scene and is folded into the per-sphere K = |c|^2 - r^2 + R^2 at upload.  What is left per sphere pair is
//       hb = fma(X, dx, fma(Y, dy, fma(Z, dz, -p.d)))          3 FFMA2
//       C  = fma(X, -2px, fma(Y, -2py, fma(Z, -2pz, K)))       3 FFMA2   (K is the chain head's addend: no separate add)
//       disc' = fma(hb, hb, -C)                                1 FFMA2
//   and one SHF per test (ALU pipe) that funnel-shifts the sign bit of disc' into a 32-sphere word.  B200 issues one
//   warp instruction per cycle per sub-partition and an FFMA2 holds the issue port for two, so the scan costs
//   14 + 2 (SHF) + 2 (LDS.128) cycles per sphere pair (tools/probe_ur.cu: 8 ops 60.7, 7 ops 65.8 TFLOP/s-equivalent).
//   The expansion cancels |c|^2 + R^2 against 2 c.p, which is why it is only a FILTER: K is lowered at upload by
//   RT_FILTER_SLACK (|c|^2 + r^2 + R^2) and p is placed slightly outside the R-sphere (|p|^2 = R^2 + sigma, sigma covering
//   the f32 error of the foot point of a distant origin), so disc' >= 0 is a conservative superset of
//   "discriminant >= 0" (sphere.rs:24-25).  Every survivor goes through the well-conditioned sphere_roots.
//   A line that misses the R-sphere can hit no small sphere; its filter ray is zeroed so that nothing passes.
//
//   Candidates (a few per ray): positions appended to a per-lane list in shared memory, then the whole warp drains its
//   lists in lock-step through candidate<float>.
//
// Table layout: one 64-byte record per 4 spheres, [cx0..3][cy0..3][cz0..3][K0..3], in list order of `small`, padded to whole
// 32-sphere words with never-hit entries plus ONE extra record (the software pipeline always loads one record ahead).
// A word is 512 contiguous bytes: every LDS.128 of the unrolled word is [base + immediate].
#define RT_TABLE_FLOATS(np) (4 * (size_t)(np) + 16)

// The line gate of both filters (this one and the tensor-core filter of rt_umma_scan.cuh): f, the foot point of the
// coordinate origin on the line, orthogonalised twice (the second pass removes the O(u |o|) component along dhat that the
// first leaves when the origin is far away); sigma = 16 u r_max |o|_1, as the foot point of a far origin is only known to
// ~4 u |o|; live: the line enters the R-sphere widened by sigma.  A line that misses it can hit no small sphere.
struct LineGate {
    V3<float> f;
    float sigma;
    bool live;
};
__device__ __forceinline__ LineGate line_gate(V3<float> o, V3<float> dhat, float inv_a, float R2, float sigma_per_len)
{
    LineGate g;
    g.f = o - dhat * (dot(o, dhat) * inv_a);
    g.f = g.f - dhat * (dot(g.f, dhat) * inv_a);
    g.sigma = sigma_per_len * (fabsf(o.x) + fabsf(o.y) + fabsf(o.z));
    g.live = length_squared(g.f) < R2 + g.sigma;
    return g;
}

struct FilterRay {
    float M2PX, M2PY, M2PZ, DX, DY, DZ, NPD;
};
__device__ __forceinline__ FilterRay make_filter_ray(V3<float> o, V3<float> dhat, float inv_a, float R2, float sigma_per_len)
{
    const LineGate g = line_gate(o, dhat, inv_a, R2, sigma_per_len);
    // |p|^2 = R^2 + sigma
    const float s = g.live ? sqrtf(((R2 + g.sigma) - length_squared(g.f)) * inv_a) : 0.0f;
    const V3<float> p = g.f - dhat * s;                     // where the line enters the R-sphere
    FilterRay r;
    // A line that misses the R-sphere (an origin far out on the ground, heading for the sky) can hit no small sphere:
    // with p = 0 the filter computes (c.d)^2 - K <= |c|^2 - (|c|^2 - r^2 + R^2) < 0 for every sphere, as R >= |c| + |r|.
    // (Keeping the foot point instead would stay conservative, but |p|^2 - R^2 would act as slack and let through every
    // sphere within that distance of the line — hundreds of false candidates per such ray.)
    const float live = g.live ? 1.0f : 0.0f;
    r.M2PX = -2.0f * live * p.x; r.M2PY = -2.0f * live * p.y; r.M2PZ = -2.0f * live * p.z;
    // opaque to the compiler: otherwise it keeps p and re-multiplies by -2 in every 32-sphere word (3 FMUL per word)
    asm volatile("" : "+f"(r.M2PX), "+f"(r.M2PY), "+f"(r.M2PZ));
    r.DX = dhat.x; r.DY = dhat.y; r.DZ = dhat.z;
    r.NPD = -live * dot(p, dhat);
    return r;
}

// One 4-sphere record of the filter: the sign bits of the 4 disc' shifted into m, the record's last sphere in bit 0.
__device__ __forceinline__ unsigned filter_record(unsigned m, float4 cx, float4 cy, float4 cz, float4 kk, const FilterRay& f)
{
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const float2 X = h ? make_float2(cx.z, cx.w) : make_float2(cx.x, cx.y);
        const float2 Y = h ? make_float2(cy.z, cy.w) : make_float2(cy.x, cy.y);
        const float2 Z = h ? make_float2(cz.z, cz.w) : make_float2(cz.x, cz.y);
        const float2 K = h ? make_float2(kk.z, kk.w) : make_float2(kk.x, kk.y);
        const float2 hb = ffma2(X, bc2(f.DX), ffma2(Y, bc2(f.DY), ffma2(Z, bc2(f.DZ), bc2(f.NPD))));
        const float2 C = ffma2(X, bc2(f.M2PX), ffma2(Y, bc2(f.M2PY), ffma2(Z, bc2(f.M2PZ), K)));
        const float2 disc = ffma2(hb, hb, neg2(C));
        m = __funnelshift_l(__float_as_uint(disc.x), m, 1);
        m = __funnelshift_l(__float_as_uint(disc.y), m, 1);
    }
    return m;
}

// One 32-sphere word of the filter: 8 records, software-pipelined one record ahead (the ~30-cycle shared-memory latency
// hides behind the 14 FFMA2 of the current record).  Bit (31-k) of the result is CLEAR when sphere k passed.
__device__ __forceinline__ unsigned filter_word(const float4* __restrict__ rec, const FilterRay& f, float4& ncx, float4& ncy, float4& ncz, float4& nkk)
{
    unsigned m = 0;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const float4 cx = ncx, cy = ncy, cz = ncz, kk = nkk;
        ncx = rec[4 * q + 4]; ncy = rec[4 * q + 5]; ncz = rec[4 * q + 6]; nkk = rec[4 * q + 7];
        m = filter_record(m, cx, cy, cz, kk, f);
    }
    return m;
}

// The last, partial word of the table: only its n_rec (1..7) records that hold real spheres are filtered (the final scene's
// 529 small spheres are 16 words + 5 records: filtering the 3 all-padding records would be 2 % of the scan for nothing).
__device__ __forceinline__ float4 ld_rec(const float4* p, unsigned saddr, int i, bool smem)
{
    if (!smem) return p[i];
    float4 v;                                               // shared-window load: a non-inlined function only sees a generic pointer
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr + 16u * (unsigned)i));
    return v;
}
template <bool kSmem>
__device__ __noinline__ unsigned filter_tail(const float4* __restrict__ rec, int n_rec, FilterRay f)
{
    unsigned m = 0;
    unsigned sa = kSmem ? (unsigned)__cvta_generic_to_shared(rec) : 0u;
    float4 ncx = ld_rec(rec, sa, 0, kSmem), ncy = ld_rec(rec, sa, 1, kSmem), ncz = ld_rec(rec, sa, 2, kSmem), nkk = ld_rec(rec, sa, 3, kSmem);
#pragma unroll 1
    for (int q = 0; q < n_rec; ++q, rec += 4, sa += 64u) {
        const float4 cx = ncx, cy = ncy, cz = ncz, kk = nkk;
        ncx = ld_rec(rec, sa, 4, kSmem); ncy = ld_rec(rec, sa, 5, kSmem); ncz = ld_rec(rec, sa, 6, kSmem); nkk = ld_rec(rec, sa, 7, kSmem);
        m = filter_record(m, cx, cy, cz, kk, f);
    }
    const int absent = 32 - 4 * n_rec;                       // spheres of the word that were not filtered: marked "not passed"
    return (m << absent) | ((1u << absent) - 1u);
}

// The precise test of small sphere p, unless it is the one the ray starts on (candidate_self tests that one).
__device__ __forceinline__ void candidate_small(const float4* __restrict__ small, int p, V3<float> o, V3<float> dhat, float inv_a, float t_min,
                                                int self_pos, float* t_best, int* p_best)
{
    if (p != self_pos) { const float4 s = small[p]; candidate<float, true>(o, dhat, inv_a, t_min, mk(s.x, s.y, s.z), s.w, p, t_best, p_best); }
}

// Candidate collection of both filters: the survivors of one pass word (bit (31-k) set: sphere p0 + k passed) go onto the lane's
// list (slot k at cand[k * stride]) as positions relative to `base`, and once the list holds RT_CAND_CAP, straight to the precise
// test.  uint16 slots: the FP32 table can hold more than 65 535 spheres, so that scan lists positions relative to its segment.
__device__ __forceinline__ void collect(unsigned pass, int p0, int base, uint16_t* cand, int stride, int* nc, const float4* __restrict__ small,
                                        V3<float> o, V3<float> dhat, float inv_a, float t_min, int self_pos, float* t_best, int* p_best)
{
    while (pass) {
        const int k = __clz(pass);
        pass &= ~(0x80000000u >> k);
        const int p = p0 + k;
        if (*nc < RT_CAND_CAP) { cand[*nc * stride] = (uint16_t)(p - base); ++*nc; }
        else candidate_small(small, p, o, dhat, inv_a, t_min, self_pos, t_best, p_best);
    }
}

template <bool kSmem>
__device__ __forceinline__ void scan_small(const float* __restrict__ table, int n_rec, float R2, float sigma_per_len, const float4* __restrict__ small,
                                           V3<float> o, V3<float> dhat, float inv_a, float t_min, int self_pos, V3<float> self_n,
                                           uint16_t* cand, int cand_stride, float* t_best, int* p_best)
{
    const int n_words = n_rec >> 3, n_tail = n_rec & 7;          // whole 32-sphere words; records of the partial last word
    int pb = *p_best; float tb = *t_best;
    // the sphere the ray starts on is tested on its own, independently of the filter
    if (self_pos >= 0) candidate_self<float>(dhat, inv_a, t_min, self_n, small[self_pos].w, self_pos, &tb, &pb);
    if (n_rec == 0) { *p_best = pb; *t_best = tb; return; }

    const FilterRay f = make_filter_ray(o, dhat, inv_a, R2, sigma_per_len);
    const float4* rec = reinterpret_cast<const float4*>(table);
    float4 ncx = rec[0], ncy = rec[1], ncz = rec[2], nkk = rec[3];
    int w0 = 0;
    do {
        const int w1 = min(w0 + RT_SEG_WORDS, n_words);
        int nc = 0;
        for (int w = w0; w < w1; ++w, rec += 32)
            collect(~filter_word(rec, f, ncx, ncy, ncz, nkk), w << 5, w0 << 5, cand, cand_stride, &nc, small, o, dhat, inv_a, t_min, self_pos, &tb, &pb);
        if (w1 == n_words && n_tail) {                                   // the partial word: survivors go straight to the precise test
            unsigned c = ~filter_tail<kSmem>(reinterpret_cast<const float4*>(table) + (size_t)n_words * 32, n_tail, f);
            while (c) {
                const int k = __clz(c);
                c &= ~(0x80000000u >> k);
                candidate_small(small, (n_words << 5) + k, o, dhat, inv_a, t_min, self_pos, &tb, &pb);
            }
        }
        const int nmax = __reduce_max_sync(RT_FULL, nc);
        for (int k = 0; k < nmax; ++k)
            if (k < nc) candidate_small(small, (w0 << 5) + cand[k * cand_stride], o, dhat, inv_a, t_min, self_pos, &tb, &pb);
        w0 = w1;
    } while (w0 < n_words);
    *p_best = pb; *t_best = tb;
}

struct HitD {            // the large spheres' closest hit, t kept in f64 for the merge
    double t;
    int idx;
    int code;
};

// The spheres too large for f32 (|oc|^2 - r^2 of sphere.rs:22 cancels: the r = 1000 ground, main.rs:64), tested in f64.
// Not inlined: rare (a lane the f32 form does not cover), and kept out of the scan's register allocation.
__device__ __noinline__ HitD big_spheres_best(const double4* __restrict__ big, const int* __restrict__ big_idx, int nb, V3<float> o, V3<float> dhat,
                                              float t_min, int self_code, V3<float> self_n)
{
    const V3<double> od = mk<double>(o.x, o.y, o.z), dd = mk<double>(dhat.x, dhat.y, dhat.z);
    const double inv_ad = 2.0 - length_squared(dd);          // 1/a for a = 1 + e, |e| < 1e-6: exact to e^2
    double tbd = __longlong_as_double(0x7ff0000000000000LL); int ib = -1, code = RT_SELF_NONE;
    for (int b = 0; b < nb; ++b) {
        const double4 s = big[b];
        const int before = ib; const double tbefore = tbd;
        if (self_code == -2 - b) {
            // self_n is unit to f32 rounding (|sn|^2 = 1 + e, |e| < 1e-6): one Newton step of 1/sqrt from the seed 1 is exact to
            // e^2 — no f64 sqrt and division (~60 instructions on a pipe that runs at 1/32 of the FP32 rate)
            V3<double> sn = mk<double>(self_n.x, self_n.y, self_n.z);
            sn = sn * (1.5 - 0.5 * length_squared(sn));
            candidate_self<double>(dd, inv_ad, (double)t_min, sn, s.w, big_idx[b], &tbd, &ib);
        } else {
            candidate<double, true>(od, dd, inv_ad, (double)t_min, mk(s.x, s.y, s.z), s.w, big_idx[b], &tbd, &ib);
        }
        if (ib != before || tbd != tbefore) code = -2 - b;
    }
    HitD h; h.t = tbd; h.idx = ib; h.code = code;
    return h;
}

// The large spheres in f32.  `half_b^2 - a c` (sphere.rs:24) cancels in f32 for a sphere of radius 1000
// because c = |o - c|^2 - r^2 is formed from two numbers of size 10^6.  Expanded around the COORDINATE origin instead,
//     C = |o|^2 - 2 o.c + K ,   K = |c|^2 - r^2  (per sphere, from f64, carried as hi + lo)
// has terms of the size of the result whenever the origin is near the scene and outside the sphere (the ground: K = 0,
// C = |o|^2 + 2000 o_y, all positive), and the roots follow without the second cancellation (tca - sqrt) as
//     q = hb + copysign(sqrt(hb^2 - a C), hb) ,  { q / a , C / q } ,   hb = (c - o).d   (c as hi + lo).
// A lane whose C does cancel (sum of |terms| > 16 |C|: origins far from the coordinate origin yet close to the surface) reports
// need64 and takes the f64 routine instead; so does every lane when a sphere's data is not exactly representable.
// ~35 FP32 instructions instead of ~45 FP64 ones on a pipe that B200 runs at 1/32 of the FP32 rate: 2000 -> 300 cycles per ray.
__device__ __forceinline__ void big_spheres_f32(const float4* __restrict__ bigf, const int* __restrict__ big_idx, int nb, V3<float> o, V3<float> dhat,
                                                float t_min, int self_code, V3<float> self_n, float* t_out, int* idx_out, int* code_out, bool* need64)
{
    const float a = length_squared(dhat), inv_a = 2.0f - a;
    const float oo = length_squared(o), od = dot(o, dhat);
    float tb = __int_as_float(0x7f800000); int ib = -1, code = RT_SELF_NONE; bool bad = false;
    for (int b = 0; b < nb; ++b) {
        const float4 q0 = bigf[3 * b], q1 = bigf[3 * b + 1], q2 = bigf[3 * b + 2];
        const int idx = big_idx[b];
        float t;
        if (self_code == -2 - b) {
            // the sphere the ray starts on: roots {0, 2 tca}, origin taken ON the surface (candidate_self)
            t = -2.0f * fabsf(q0.w) * dot(self_n, dhat) * inv_a;
            if (!(t >= t_min)) continue;
        } else {
            const V3<float> ch = mk(q0.x, q0.y, q0.z), cl = mk(q1.x, q1.y, q1.z);
            const float P = dot(o, ch) + dot(o, cl);
            const float C = (oo - 2.0f * P + q1.w) + q2.x;
            bad |= (oo + 2.0f * fabsf(P) + fabsf(q1.w)) > 16.0f * fabsf(C);
            const float hb = (dot(ch, dhat) - od) + dot(cl, dhat);
            const float disc = hb * hb - a * C;
            if (disc < 0.0f) continue;                                    // sphere.rs:25
            const float sq = sqrtf(disc);
            const float qq = hb + copysignf(sq, hb);
            const float r0 = qq * inv_a, r1 = C / qq;                      // the two roots (qq == 0 only when hb == C == 0: origin on the surface, tangent)
            const float t1 = fminf(r0, r1), t2 = fmaxf(r0, r1);
            t = t1;                                                        // sphere.rs:28
            if (!(t >= t_min)) { t = t2; if (!(t >= t_min)) continue; }   // sphere.rs:29-33 with t_max = +inf
        }
        if (t < tb || (t == tb && idx > ib)) { tb = t; ib = idx; code = -2 - b; }
    }
    *t_out = tb; *idx_out = ib; *code_out = code; *need64 = bad;
}

// The large spheres' own closest hit: the f32 form, or f64 for the lanes / scenes it does not cover.
__device__ __forceinline__ HitD big_spheres(const float4* __restrict__ bigf, const double4* __restrict__ big, const int* __restrict__ big_idx, int nb,
                                            V3<float> o, V3<float> dhat, float t_min, int self_code, V3<float> self_n)
{
    bool need64 = bigf == nullptr;
    HitD h; float tf = __int_as_float(0x7f800000); h.idx = -1; h.code = RT_SELF_NONE;
    if (!need64) big_spheres_f32(bigf, big_idx, nb, o, dhat, t_min, self_code, self_n, &tf, &h.idx, &h.code, &need64);
    h.t = (double)tf;
    if (need64) h = big_spheres_best(big, big_idx, nb, o, dhat, t_min, self_code, self_n);
    return h;
}

// The large spheres' hit merged into the small spheres' one by (t ascending, list index descending), sphere.rs:29,31 +
// mod.rs:61-66, compared in f64.  A total order: the winner is the one a test of the large spheres seeded with h would give.
__device__ __forceinline__ HitF merge_big(HitF h, HitD b)
{
    if (b.idx >= 0 && (b.t < (double)h.t || (b.t == (double)h.t && b.idx > h.idx))) { h.t = (float)b.t; h.idx = b.idx; h.code = b.code; }
    return h;
}

// The FP32 scan's call.  Not inlined: once per ray, and kept out of the filter loop's register allocation.
__device__ __noinline__ HitF big_spheres_merge(const float4* __restrict__ bigf, const double4* __restrict__ big, const int* __restrict__ big_idx, int nb,
                                               V3<float> o, V3<float> dhat, float t_min, int self_code, V3<float> self_n, HitF h)
{
    return merge_big(h, big_spheres(bigf, big, big_idx, nb, o, dhat, t_min, self_code, self_n));
}

// Closest hit of one ray against the whole scene: HittableList::hit (mod.rs:56-69).
// float: packed filter over the small spheres + f64 test of the big ones; all lanes of the warp
// must call together.  self_code / self_n identify the sphere the ray starts on (RT_SELF_NONE for
// camera rays).  Returns t in dhat units, the list index (or -1) and the winner's code.
template <bool kSmem>
__device__ __forceinline__ HitF closest_hit(const SceneDev& sc, const float* table, V3<float> o, V3<float> dhat, float t_min,
                                            int self_code, V3<float> self_n, uint16_t* cand, int cand_stride)
{
    const float inv_a = 2.0f - length_squared(dhat);           // 1/a for a = 1 + e, |e| < 1e-6 (dhat is unit to rounding): exact to e^2, no MUFU.RCP
    float tb = __int_as_float(0x7f800000);   // f64::INFINITY at main.rs:44
    int pb = -1;
    scan_small<kSmem>(table, sc.n_rec, sc.filter_R2, sc.filter_sigma, sc.small, o, dhat, inv_a, t_min, self_code, self_n, cand, cand_stride, &tb, &pb);
    HitF h; h.t = tb; h.idx = pb >= 0 ? sc.small_idx[pb] : -1; h.code = pb;
    if (sc.nb > 0) h = big_spheres_merge(sc.bigf, sc.big, sc.big_idx, sc.nb, o, dhat, t_min, self_code, self_n, h);
    return h;
}

// double: the reference's arithmetic width, every sphere through the precise test (triage mode).
// code == list index here.
__device__ __forceinline__ void closest_hit_f64(const SceneDev& sc, V3<double> o, V3<double> dhat, double t_min, int self_idx, V3<double> self_n,
                                                double* t_out, int* idx_out)
{
    const double inv_a = 1.0 / length_squared(dhat);
    double tb = __longlong_as_double(0x7ff0000000000000LL);
    int ib = -1;
    for (int i = 0; i < sc.n; ++i) {
        const double4 s = sc.sphd[i];
        if (i == self_idx) candidate_self<double>(dhat, inv_a, t_min, self_n, s.w, i, &tb, &ib);
        else candidate<double>(o, dhat, inv_a, t_min, mk(s.x, s.y, s.z), s.w, i, &tb, &ib);
    }
    *t_out = tb; *idx_out = ib;
}

// Dynamic shared memory of every scanning kernel: [candidate lists: threads x RT_CAND_CAP uint16][filter table].
// The lists come first so that a lane's slot address does not depend on the scene size.  Returns the table to scan
// (the staged copy, or the global one when kSmem is false) and the lane's first list slot (slot k at cand[k * threads]).
#define RT_CAND_BYTES(threads) ((size_t)(threads) * RT_CAND_CAP * sizeof(uint16_t))
template <bool kSmem>
__device__ __forceinline__ const float* setup_scan_smem(unsigned char* smem_raw, const SceneDev& sc, int threads, uint16_t** cand)
{
    *cand = reinterpret_cast<uint16_t*>(smem_raw) + threadIdx.x;
    if (!kSmem) return sc.table;
    float4* dst = reinterpret_cast<float4*>(smem_raw + RT_CAND_BYTES(threads));
    const float4* src = reinterpret_cast<const float4*>(sc.table);
    const int n4 = (int)(RT_TABLE_FLOATS(sc.np) / 4);
    for (int i = threadIdx.x; i < n4; i += threads) dst[i] = src[i];          // cooperative 16-byte copies
    __syncthreads();
    return reinterpret_cast<const float*>(dst);
}

}  // namespace rt
