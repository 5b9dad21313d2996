// rt_umma_scan.cuh — HittableList::hit (/root/reference/src/shapes/mod.rs:56-69) with the sphere filter on the tensor cores.
//
// CTA = G ray groups of 128 threads (4 warps: warp q of a group owns TMEM lanes [32q, 32q+32)) + G issuer warps.
// One scan of a group = 128 rays against every small sphere of the scene:
//   ray threads   : the ray's two rows (rt_umma.cuh, ray_rows) -> tcgen05.st into the group's A columns -> arrive(a_full, mbarrier)
//   issuer warp   : wait(a_full); per chunk of NC spheres: bar.sync(hand-back) ; 2 x tcgen05.mma (row2 . B2, then row1 . B1) into
//                   the group's D columns (fp16 accumulator) ; tcgen05.commit -> full (mbarrier)
//   ray threads   : wait(full) ; tcgen05.ld.pack::16b their own lane: NC discriminants of THEIR ray, two per register ;
//                   bar.arrive(hand-back) ; sign bits -> 32-sphere words, four per instruction (sign_word16) ; survivors ->
//                   per-lane candidate list (collect, shared with the FP32 scan of rt_scene.cuh) -> precise test
//                   (sphere_roots, rt_device.cuh).
// The issuer is a warp of its own because tcgen05.mma issue stalls the issuing thread while the tensor pipe is busy
// (tools/probe_umma_filter.cu: an issuer that shares a warp with an epilogue halves the throughput), and every group has
// its own: one thread polling all groups' barriers (mbarrier.test_wait) measured 40 % slower in situ.  D is single-buffered
// per group: while one group's MMAs run, the other groups collect signs, so the tensor pipe and the ALU pipe overlap across
// groups.  The render kernel is bound by latency chains — the per-chunk round trip and the per-ray code — and every extra group
// hides more of them (G = 4 -> 6: +13 %), so G is as large as TMEM allows: 6 x (64 + 16) = 480 of 512 columns (what was
// measured around this shape is in DESIGN.md §1.2 and §7.1).
// Each CTA owns all 512 TMEM columns, so exactly one CTA may live on an SM: the launch asks for more than half of the
// SM's shared memory.
#pragma once
#include "rt_scene.cuh"
#include "rt_umma.cuh"

namespace rt {

#ifndef RT_UMMA_GROUPS
#define RT_UMMA_GROUPS 6                      // ray groups per CTA in the product kernels (24 ray warps + 6 issuer warps = 960 threads; the render kernel pads to 1024)
#endif
#ifndef RT_UMMA_CHUNK
#define RT_UMMA_CHUNK 64                      // spheres per MMA chunk (TMEM: 6 x (64 + 16) = 480 of 512 columns)
#endif
#ifndef RT_UMMA_AFULL_BACKOFF_NS
#define RT_UMMA_AFULL_BACKOFF_NS 0            // the issuer's sleep between polls while its group is in the per-ray phase (0, 100, 400 ns measured the same)
#endif
#ifndef RT_UMMA_RAY_REGS
#define RT_UMMA_RAY_REGS 72                   // setmaxnreg of the render kernel's ray warpgroups ...
#define RT_UMMA_ISSUER_REGS 32                // ... and of its issuer warpgroups (launch bound: 64)
#endif
#ifndef RT_UMMA_DRAIN_ILP
#define RT_UMMA_DRAIN_ILP 3                   // survivors per lane per lock-step round of the precise test (2: -0.2 %, 4: -0.4 %)
#endif
#define RT_UMMA_MIN_SMEM (120 * 1024)        // > half an SM's shared memory: one CTA per SM (each CTA allocates all of TMEM)

template <int G, int NC> struct UmmaShape {
    static_assert(NC % 32 == 0 && NC >= 32 && NC <= 256, "chunk = whole 32-sphere words");
    static constexpr int kRayThreads = G * 128, kThreads = G * 160;
    // the render kernel re-balances registers between its ray warps and its issuer warps (setmaxnreg works on whole warpgroups of
    // 128 threads), so it is launched with the issuer side padded to a whole warpgroup; the padding warps only take part in the
    // set-up and tear-down barriers
    static constexpr int kRenderThreads = (kThreads + 127) / 128 * 128;
    static constexpr int kCols = NC + 16;                        // TMEM columns per group: D (NC) + the rays' row1 (8) + row2 (8)
    static_assert(G * kCols <= 512, "TMEM has 512 columns");
    static_assert(G <= 6, "named barriers: 0 = __syncthreads, 1..G the groups' votes, 7..6+G their hand-back barriers");
    static constexpr size_t kCandBytes = (size_t)kRayThreads * RT_CAND_CAP * sizeof(uint16_t);
    __host__ __device__ static constexpr size_t b_offset_bytes() { return (kCandBytes + 127) & ~(size_t)127; }
    __host__ __device__ static size_t bars_offset_bytes(int npad) { return b_offset_bytes() + 2 * RT_UMMA_B_BLOCK_BYTES(npad); }
    __host__ __device__ static size_t smem_bytes(int npad)
    {
        const size_t need = bars_offset_bytes(npad) + (size_t)G * 8 * 8 + 16 + (size_t)G * 4;
        return need > RT_UMMA_MIN_SMEM ? need : (size_t)RT_UMMA_MIN_SMEM;
    }
};

// Debug builds only (-DRT_UMMA_TRACE, tools/umma_trace.py): clock stamps of block 0, warp 0 for the first iterations of the render
// loop, so that the phases of an iteration (work assignment, group vote, per-ray code, feature rows, large spheres, each chunk's
// wait / load / sign collection, candidate drain) can be read off in cycles.
#ifdef RT_UMMA_TRACE
__device__ long long g_umma_trace[4096];
__device__ int g_umma_trace_n;
#define RT_STAMP(tag) do { if (blockIdx.x == 0 && threadIdx.x == 0) { int i_ = g_umma_trace_n; if (i_ < 2040) { g_umma_trace[2 * i_] = (tag); g_umma_trace[2 * i_ + 1] = clock64(); g_umma_trace_n = i_ + 1; } } } while (0)
#else
#define RT_STAMP(tag) do { } while (0)
#endif

// per-thread view of its group's resources
struct UmmaCtx {
    uint32_t t_d, t_a;              // TMEM columns of the group's D and A (row1 at t_a, row2 at t_a + 8); lane field 0
    uint32_t lane_base;             // this warp's TMEM lane quarter, in the address's lane field
    uint32_t bar_afull, bar_full;   // mbarriers: the group's 128 rows are in TMEM / the chunk's MMAs have completed (tcgen05.commit)
    uint32_t s_hi, s_lo;            // shared-window addresses of the B image's two K blocks
    uint32_t full_phase;            // parity of the next phase of `full` to wait for
    int n_chunks;
    int group, tid_in_group;
    bool issuer_warp;
    volatile int* quit;             // the group's "no more scans" flag, read by its issuer after a_full
    uint16_t* cand;                 // this lane's first candidate slot (slot k at cand[k * kRayThreads])
};

// All threads of the CTA.  Stages the B image, initialises the groups' mbarriers, allocates TMEM.
template <int G, int NC>
__device__ __forceinline__ UmmaCtx umma_setup(unsigned char* smem_raw, const SceneDev& sc, uint32_t* tmem_base_out)
{
    using S = UmmaShape<G, NC>;
    using namespace umma;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    unsigned char* b_img = smem_raw + S::b_offset_bytes();
    const size_t blk = RT_UMMA_B_BLOCK_BYTES(sc.u_npad);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + S::bars_offset_bytes(sc.u_npad));       // [G][8]: a_full, full
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + G * 8);
    int* quit = reinterpret_cast<int*>(tmem_slot + 4);
    for (size_t i = (size_t)tid * 16; i < 2 * blk; i += (size_t)blockDim.x * 16)
        *reinterpret_cast<uint4*>(b_img + i) = *reinterpret_cast<const uint4*>(sc.u_bimg + i);
    if (tid == 0) {
        for (int i = 0; i < G; ++i) {
            mbar_init(smem_u32(bars + 8 * i + 0), 128);       // every ray thread of the group
            mbar_init(smem_u32(bars + 8 * i + 1), 1);         // tcgen05.commit
            quit[i] = 0;
        }
        fence_mbar_init();
    }
    __syncwarp();
    if (warp == 0) { tmem_alloc(smem_u32(tmem_slot), 512); tmem_relinquish(); }
    fence_proxy_async_smem();                    // B was written with generic stores; the tensor core reads it through the async proxy
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    *tmem_base_out = tmem_base;

    UmmaCtx ux;
    ux.issuer_warp = warp >= 4 * G;
    ux.group = ux.issuer_warp ? warp - 4 * G : warp >> 2;
    ux.tid_in_group = ux.issuer_warp ? lane : (tid & 127);
    ux.t_d = tmem_base + (uint32_t)(ux.group * S::kCols);
    ux.t_a = ux.t_d + NC;
    ux.lane_base = (uint32_t)(32 * (warp & 3)) << 16;
    ux.bar_afull = smem_u32(bars + 8 * ux.group); ux.bar_full = ux.bar_afull + 8;
    ux.s_hi = smem_u32(b_img); ux.s_lo = ux.s_hi + (uint32_t)blk;
    ux.full_phase = 0;
    ux.n_chunks = sc.u_npad / NC;
    ux.quit = quit + ux.group;
    ux.cand = reinterpret_cast<uint16_t*>(smem_raw) + (ux.issuer_warp ? 0 : tid);
    // every one of these is the same in all lanes of a warp; broadcasting them from lane 0 tells the compiler so, and it keeps
    // TMEM addresses and barrier addresses in uniform registers (LDTM / STTM / SYNCS take them from there)
    ux.t_d = __shfl_sync(RT_FULL, ux.t_d, 0); ux.t_a = __shfl_sync(RT_FULL, ux.t_a, 0); ux.lane_base = __shfl_sync(RT_FULL, ux.lane_base, 0);
    ux.bar_afull = __shfl_sync(RT_FULL, ux.bar_afull, 0); ux.bar_full = ux.bar_afull + 8;
    ux.n_chunks = __shfl_sync(RT_FULL, ux.n_chunks, 0);
    return ux;
}

// The group's MMA issuer.  The whole warp runs the loop and one elected lane issues: every value the loop touches is broadcast
// from lane 0 first, so the compiler keeps addresses, descriptors and counters in UNIFORM registers — tcgen05.mma takes its
// operands from there, and a loop run by a single lane of a diverged warp pays an ELECT + four R2UR.BROADCAST + two PLOP3 per
// MMA to get them there (75 instructions per chunk; the issuers were 40 % of the issue slots of the scan phase).
// Returns when the group's ray threads have called umma_group_quit.
template <int G, int NC>
__device__ __forceinline__ void umma_issuer(const UmmaCtx& ux)
{
    using namespace umma;
    const uint32_t t_d = __shfl_sync(RT_FULL, ux.t_d, 0), t_a = __shfl_sync(RT_FULL, ux.t_a, 0);
    const uint32_t bar_afull = __shfl_sync(RT_FULL, ux.bar_afull, 0), bar_full = bar_afull + 8u;
    const uint32_t s_hi = __shfl_sync(RT_FULL, ux.s_hi, 0), s_lo = __shfl_sync(RT_FULL, ux.s_lo, 0);
    const int n_chunks = __shfl_sync(RT_FULL, ux.n_chunks, 0);
    const int group = __shfl_sync(RT_FULL, ux.group, 0);
    const uint32_t idesc = make_idesc_f16_f16(NC);
    const uint64_t dh0 = make_smem_desc(s_hi, RT_UMMA_B_LBO, RT_UMMA_B_SBO), dl0 = make_smem_desc(s_lo, RT_UMMA_B_LBO, RT_UMMA_B_SBO);
    constexpr uint32_t kStep = ((uint32_t)(NC / 8) * RT_UMMA_B_SBO) >> 4;     // descriptor start-address units (16 bytes) per chunk
    uint32_t a_phase = 0; bool used = false;
    for (;;) {
        mbar_wait(bar_afull, a_phase, RT_UMMA_AFULL_BACKOFF_NS); a_phase ^= 1u;   // all 128 feature rows are in TMEM — or the group is done
        if (*ux.quit) break;
        tc_fence_after();
        uint64_t dh = dh0, dl = dl0;                                           // the chunk's B descriptors, stepped after the issue so that
#pragma unroll 1                                                               // nothing but the MMAs stands between the barrier and the tensor pipe
        for (int c = 0; c < n_chunks; ++c) {
            if (used) { named_bar_sync(7 + group, 160); tc_fence_after(); }       // the previous chunk's D has been read (umma_hand_back)
            used = true;
            if (elect_one()) {
                mma_f16_ts(t_d, t_a + 8u, dl, idesc, 0u);                 // row2 . B2: the cross terms (small: the fp16 rounding of the
                mma_f16_ts(t_d, t_a, dh, idesc, 1u);                      // intermediate D costs ~2^-12 of THEM); row1 . B1: all of hi.hi
                tc_commit(bar_full);
            }
            __syncwarp();
            dh += kStep; dl += kStep;
        }
    }
}

// group-wide OR of a predicate over the 128 ray threads (one named barrier per group)
__device__ __forceinline__ bool umma_group_any(const UmmaCtx& ux, bool pred) { return umma::named_bar_or(1 + ux.group, 128, pred); }
// every ray thread of the group, once, after its last scan: releases the group's issuer
__device__ __forceinline__ void umma_group_quit(const UmmaCtx& ux)
{
    if (ux.tid_in_group == 0) *ux.quit = 1;
    umma::mbar_arrive(ux.bar_afull);             // release; the issuer's wait acquires and then reads the flag
}
// all threads of the CTA, last thing
__device__ __forceinline__ void umma_teardown(uint32_t tmem_base)
{
    umma::tc_fence_before();
    __syncthreads();
    if ((threadIdx.x >> 5) == 0) umma::tmem_dealloc(tmem_base, 512);
}

// a ray warp is done with the chunk's D.  The issuer waits for the group's four warps on a NAMED barrier (ids 7..12, 128 ray
// threads arriving + the issuer warp syncing): the hardware wakes it on the last arrival, where an mbarrier poll loop costs a
// round of try_wait / branch instructions before the MMAs of the next chunk go out — and that hop is on the scan's critical
// path (ray rows -> MMA -> commit -> TMEM load -> hand back -> MMA ...: ~900 cycles per chunk for ~90 cycles of tensor work)
__device__ __forceinline__ void umma_hand_back(const UmmaCtx& ux)
{
    umma::named_bar_arrive(7 + ux.group, 160);
}

// Closest hit of one ray against the whole scene — the tensor-core twin of closest_hit<kSmem> (rt_scene.cuh); every one of
// the group's 128 ray threads must call together (lanes without a ray pass anything: their result is ignored).
// `has_ray`: this lane carries a ray.  A warp without any (the end of a frame: the queue is empty and its paths are done, while
// a neighbour's 50-bounce path keeps the group scanning) only keeps the group's barriers moving — no feature rows, no TMEM
// loads, no sign collection — so that the warps that still work get the SM to themselves and the frame's tail gets shorter.
template <int G, int NC>
__device__ __forceinline__ HitF closest_hit_umma(UmmaCtx& ux, const SceneDev& sc, V3<float> o, V3<float> dhat, float t_min, int self_code, V3<float> self_n,
                                                 bool has_ray = true)
{
    using namespace umma;
    if (!__any_sync(RT_FULL, has_ray)) {
        tc_fence_before();
        mbar_arrive(ux.bar_afull);                                         // (the rows this warp left in A belong to nobody: their D rows are never read)
        for (int c = 0; c < ux.n_chunks; ++c) {
            mbar_wait_spin(ux.bar_full, ux.full_phase); ux.full_phase ^= 1u;
            tc_fence_after();
            tc_fence_before();
            umma_hand_back(ux);
        }
        HitF none; none.t = __int_as_float(0x7f800000); none.idx = -1; none.code = RT_SELF_NONE;
        return none;
    }
    constexpr int kStride = UmmaShape<G, NC>::kRayThreads;
    const float inv_a = 2.0f - length_squared(dhat);           // 1/a for a = 1 + e, |e| < 1e-6
    float tb = __int_as_float(0x7f800000);                     // f64::INFINITY at main.rs:44
    int pb = -1;
    // the sphere the ray starts on is tested on its own, independently of the filter (rt_scene.cuh, candidate_self)
    if (self_code >= 0) candidate_self<float>(dhat, inv_a, t_min, self_n, sc.small[self_code].w, self_code, &tb, &pb);

    {
        const LineGate g = line_gate(o, dhat, inv_a, sc.filter_R2, sc.filter_sigma);
        uint32_t row1[8], row2[8];
        ray_rows(g.f.x, g.f.y, g.f.z, dhat.x, dhat.y, dhat.z, g.live, g.sigma, sc.u_sc, row1, row2);
        tmem_st8(ux.t_a + ux.lane_base, row1);
        tmem_st8(ux.t_a + 8u + ux.lane_base, row2);
    }
    tc_wait_st();
    tc_fence_before();
    mbar_arrive(ux.bar_afull);
    RT_STAMP(5);

    // the large spheres while the first chunk's MMAs are in flight (later, inside the chunk loop, they delay the warp's hand-backs:
    // DESIGN.md §7.1)
    HitD big{__longlong_as_double(0x7ff0000000000000LL), -1, RT_SELF_NONE};
    if (sc.nb > 0) big = big_spheres(sc.bigf, sc.big, sc.big_idx, sc.nb, o, dhat, t_min, self_code, self_n);

    RT_STAMP(6);
    int nc = 0;
    for (int c = 0; c < ux.n_chunks; ++c) {
        mbar_wait_spin(ux.bar_full, ux.full_phase); ux.full_phase ^= 1u;
        RT_STAMP(10 + c);
        tc_fence_after();
        uint32_t v[NC / 32][16];
#pragma unroll
        for (int w = 0; w < NC / 32; ++w) tmem_ld16p(ux.t_d + ux.lane_base + 32u * w, v[w]);
        tc_wait_ld();
        RT_STAMP(40 + c);
        tc_fence_before();                                                     // hand D back to the issuer, whose next MMAs then
        umma_hand_back(ux);                                                    // overlap the sign collection
#pragma unroll
        for (int w = 0; w < NC / 32; ++w)                                      // ~sign_word16: bit (31-k) set when sphere k passed
            collect(~sign_word16(v[w]), c * NC + w * 32, 0, ux.cand, kStride, &nc, sc.small, o, dhat, inv_a, t_min, self_code, &tb, &pb);
        RT_STAMP(70 + c);
    }
    RT_STAMP(7);
    // survivors through the precise test, the warp in lock step, RT_UMMA_DRAIN_ILP per round: the test is one dependent chain (load,
    // ~25 FP operations, a MUFU), so independent ones per lane divide the rounds' latency (the drain is 11 % of an iteration); all of
    // a round's list reads and sphere loads are issued before its first test (that alone was worth 2 %).  The FP32 scan's drain
    // (scan_small) is kept apart: this form, at one survivor per round, compiles to longer code there.
    const int nmax = __reduce_max_sync(RT_FULL, nc);
    for (int k = 0; k < nmax; k += RT_UMMA_DRAIN_ILP) {
        int pp[RT_UMMA_DRAIN_ILP]; bool gg[RT_UMMA_DRAIN_ILP]; float4 ss[RT_UMMA_DRAIN_ILP];
#pragma unroll
        for (int j = 0; j < RT_UMMA_DRAIN_ILP; ++j) {
            const bool h = k + j < nc;
            pp[j] = h ? ux.cand[(k + j) * kStride] : self_code;
            gg[j] = h && pp[j] != self_code;
        }
#pragma unroll
        for (int j = 0; j < RT_UMMA_DRAIN_ILP; ++j) ss[j] = gg[j] ? sc.small[pp[j]] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int j = 0; j < RT_UMMA_DRAIN_ILP; ++j)
            if (gg[j]) candidate<float, true>(o, dhat, inv_a, t_min, mk(ss[j].x, ss[j].y, ss[j].z), ss[j].w, pp[j], &tb, &pb);
    }
    RT_STAMP(8);
    HitF h; h.t = tb; h.idx = pb >= 0 ? sc.small_idx[pb] : -1; h.code = pb;
    return merge_big(h, big);
}

}  // namespace rt
