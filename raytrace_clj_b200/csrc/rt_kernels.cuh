// rt_kernels.cuh — sm_100a kernels of libraytrace_b200.so.
//
//   Culler<R,BLOCK,COMMON>  the hot loop: brute-force FP32 cull of R rays per thread against the sphere list staged in
//                      shared memory (Hitlist.hit?, hitable.clj:15-26); the survivors' sign bits go, branch-free, to
//                      per-thread mask words in shared memory.  COMMON: the cheaper form for rays that share an origin.
//   SurvivorIter       walks the mask words that hold a survivor
//   RefineSink         survivors refined in FP64 by the owning thread (trace kernel, megakernel)
//   PairSink           survivors emitted as (ray, sphere) pairs for the pooled FP64 refine (wavefront kernels)
//   wf_generate / wf_cull / wf_refine / wf_tiebreak / wf_shade / wf_tail
//                      wavefront path tracer (pixel + color, core.clj:17-57): one kernel per stage over a queue of
//                      paths; wf_cull is the hot-loop kernel, wf_tail finishes the last short iterations CTA by CTA
//   mega_kernel        persistent megakernel with per-lane path regeneration, kept for comparison
//   trace_kernel       closest hit of caller-given rays (rt_trace_primary)
//   cull_check_kernel / shade_kernel / genrays_kernel   diagnostics for the parity tests
//   resolve_kernel     core.clj:52-57 + the y flip of core.clj:105 (+ NVLink peer reduce)
//   ffma_peak_kernel   FP32 roofline denominator measured on the box
#pragma once

#include "rt_device.cuh"

namespace rt {

#define RT_FOR_R _Pragma("unroll") for (int r = 0; r < R; ++r)

// one logged ray of rt_trace_paths (= rt_path_bounce of the C ABI)
struct PathBounce {
    float o[3];
    float time;
    float d[3];
    int hit_id;
    double t;
};

struct RenderParams {
    DevScene sc;
    DevCamera cam;
    int nx, ny;
    int sample_begin, sample_count;
    int row_offset, row_stride, rows_in_shard;
    int max_depth;
    uint2 key;
    float* sum;                           // nx*ny*3, += ; pixel (i, j) at (j*nx+i)*3, j = 0 bottom
    unsigned long long* counters;         // DC_COUNT
    unsigned long long* work_counter;     // next (sample, pixel) work item
    unsigned long long total_work;        // sample_count * nx * rows_in_shard
    int cull_cap;                         // float4 slots of the shared-memory sphere tile
    int preloaded;                        // 1: whole scene fits one tile (loaded once per CTA)
    int common_origin;                    // 1: every camera ray starts at cam.origin (pinhole, or aperture 0)
    // rt_render_views: the frame stacks n_views images of nx x ny; stacked row j_g is row j_g - v * ny of view
    // v = j_g / ny, rendered through views[v] (P.cam = views[0]).  Null / 0 = the single camera in `cam`.
    // A queue record's pixel field carries a TAG: the view-local Philox pixel in the low view_bits bits, the view above
    // them, so that every bounce reads its Philox pixel with one AND (rng_pixel) and only the sample's RED.ADD rebuilds
    // the frame slot (v * view_px + pixel, frame_slot).  A single render has view_mask = ~0, view_bits = 31, view_px = 0:
    // the tag is the frame slot.  make_path splits a frame slot as umulhi(2 slot, view_magic) >> view_shift
    // (= slot / view_px for every slot below 2^31).
    const DevCamera* views;               // [n_views]
    int n_views;
    uint32_t view_px, view_mask, view_bits, view_magic, view_shift;   // view_px = nx * ny
    // rt_trace_paths: work item w IS path w of a caller-given list instead of the w-th (sample, pixel) of the frame;
    // the queue record's "pixel" field then holds w, `sum` has 3 floats per PATH, and the path's counters / bounce log
    // are kept per path.  All null / 0 in a render.
    const int* path_pixel;                // [total_work] j * nx + i
    const int* path_sample;               // [total_work]
    int* path_nrays;                      // [total_work]
    int* path_term;                       // [total_work]
    PathBounce* path_log;                 // [total_work * path_log_n] or null
    int path_log_n;
};

// the view of a stacked frame slot (rt_render_views)
__device__ __forceinline__ uint32_t view_of(const RenderParams& P, uint32_t slot) {
    return __umulhi(slot << 1, P.view_magic) >> P.view_shift;
}
// the Philox "pixel" of the path whose queue record carries `tag` in its pixel field: a view's paths are keyed by the
// view-local pixel, exactly as a single render of that camera keys them.  VIEWS = false (the instantiations that single
// renders and rt_trace_paths run): the tag is the frame slot, and none of the batch arithmetic is compiled in.
template <bool VIEWS>
__device__ __forceinline__ uint32_t rng_pixel(const RenderParams& P, uint32_t tag) {
    return P.path_pixel ? (uint32_t)__ldg(&P.path_pixel[tag]) : (VIEWS ? tag & P.view_mask : tag);
}
// the frame slot (the path of rt_trace_paths) a queue record's tag adds its radiance to
template <bool VIEWS>
__device__ __forceinline__ uint32_t frame_slot(const RenderParams& P, uint32_t tag) {
    return VIEWS ? (tag & P.view_mask) + (tag >> P.view_bits) * P.view_px : tag;
}
// rt_trace_paths bookkeeping for ray number `ray_no` (0-based) of path `slot`
__device__ __forceinline__ void path_log_ray(const RenderParams& P, uint32_t slot, int ray_no, float4 a, float4 b, int k, double t) {
    if (P.path_log && ray_no < P.path_log_n) {
        PathBounce& L = P.path_log[(size_t)slot * P.path_log_n + ray_no];
        L.o[0] = a.x; L.o[1] = a.y; L.o[2] = a.z; L.time = a.w;
        L.d[0] = b.x; L.d[1] = b.y; L.d[2] = b.z;
        L.hit_id = k < 0 ? -1 : __ldg(&P.sc.orig_id[k]);
        L.t = t;
    }
}
__device__ __forceinline__ void path_log_end(const RenderParams& P, uint32_t slot, int n_rays, int reason) {
    if (P.path_nrays) {
        P.path_nrays[slot] = n_rays;
        P.path_term[slot] = reason;
    }
}

// exact test of (ray, leaf k): the sphere formula, or the generic leaves of a scene marshalled through rt_set_scene_ex.
// path context (for the `rand` of a ConstantMedium): Philox key / pixel / sample / bounce, or has_ctx = false (u = 0.5).
template <bool GEN>
__device__ __forceinline__ double refine_leaf(const DevScene* sc, int k, float ox, float oy, float oz, float dx, float dy, float dz,
                                              float time, double tmin, double tmax, bool has_ctx, uint2 key, uint32_t pixel,
                                              uint32_t sample, uint32_t bounce) {
    if (!GEN)
        return refine_candidate(sc->ex_c0r, sc->ex_c1, sc->ex_t0t1, sc->flags, k, ox, oy, oz, dx, dy, dz, time, tmin, tmax);
    float mu = 0.5f;
    if (has_ctx && __ldg(&sc->prim_type[k]) == PRIM_MEDIUM) mu = medium_uniform(key, pixel, sample, bounce, __ldg(&sc->orig_id[k]));
    return refine_generic(sc, k, ox, oy, oz, dx, dy, dz, time, tmin, tmax, mu);
}

// ------------------------------------------------------------------------------------------
// Culler: the FP32 test, per (ray, sphere), 9 FP32-pipe instructions (8 FFMA + 1 FADD) + 1 funnel shift.  The 17-flop
// test of SURVEY §8(d) is evaluated in expanded form so that everything that depends on the ray alone
// or on the sphere alone is hoisted (f = o - c never materialises):
//     b   = o.h - c.h                     3 FFMA   seeded with the ray's  P = o.h
//     s   = (r2i - c.c) + 2 o.c           3 FFMA   seeded with the sphere's W = r2i - c.c, ray holds m = -2 o
//     nc  = s - |o|^2                     1 FADD   ray holds Q = |o|^2 (deflated, see below)
//     key = b * min(b, 0) + nc            2 FFMA   (c c - c |c| with c = b / sqrt 2; see key_bits)
// with h = d * sqrt(1+eps) / |d| (a = d.d folded in).  key >= 0  <=>  (approaching and discriminant
// >= 0) or (origin inside the sphere): exactly the spheres that can have a root in front of the
// origin.  Rounding: with u = 2^-24 the computed key differs from the exact one by at most
// u (33.6 |o|^2 + 33.6 |c|^2 + 4.1 r2i) (DESIGN.md "Precision"); the ray's share is taken off Q
// (Q = |o|^2 (1 - 54 u)), the sphere's share is added to W on the host, so the cull only ever
// over-reports.  tests/test_gpu_parity.py::test_cull_never_under_reports checks exactly that.
// No branch and no compaction in the loop: the sign bits of a ray's keys are funnel-shifted into one
// 32-bit mask per GROUP = 32 spheres, stored at a position that implies (group, ray).  The Sink
// walks the masks of the groups flagged in a per-thread bitmap after every chunk of <= 512 spheres.
// ------------------------------------------------------------------------------------------
// 128-bit shared-memory load from a 32-bit shared-window address (keeps ptxas from re-deriving the
// generic->shared base every iteration: S2UR/UMOV/UIADD3/ULEA/LEA per sphere pair in the profile)
__device__ __forceinline__ float4 lds128(unsigned addr) {
    float4 v;
    asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ unsigned smem_addr(const void* p) {
    unsigned a = (unsigned)__cvta_generic_to_shared(p);
    asm volatile("" : "+r"(a));   // opaque: one register, not rematerialised
    return a;
}

// slice `part` of `parts` of [0, n)
__device__ __forceinline__ int slice_lo(int n, int part, int parts) { return (int)(((long long)n * part) / parts); }

constexpr int GROUP = 32;                      // spheres per mask word
constexpr int CHUNK_GROUPS = 16;               // mask words per ray between two sink flushes
constexpr int CHUNK = GROUP * CHUNK_GROUPS;    // 512 spheres
constexpr int CULL_PAD = 8;                    // the cull records are padded to a multiple of this (inner unroll)
constexpr float RAY_DEFLATE = 1.0f - 3.2e-6f;  // 1 - 54 u: the ray's share of the rounding budget, taken off |o|^2

// mask words of a thread: word (group g, ray r) at list[(g * R + r) * BLOCK + threadIdx.x] (one bank per lane).
// Bit layout: sphere j of a group of m spheres (m = 32, or the remainder in the last group of a chunk) is at
// bit m - 1 - j; a CLEAR bit = that (ray, sphere) pair survived the cull; bits >= m are set.
// COMMON = true: every ray of the batch starts at the SAME origin (camera rays of a pinhole or zero-aperture
// camera, 39 % of all rays on the random scene).  Then s - Q = (W + 2 o.c) - |o|^2 depends on the sphere only: it
// is computed once per sphere per kernel (common_record) and stored in the record's 4th component, and the test
// shrinks to the 3-FFMA chain of c plus the 2 key FFMAs: 5 FP32 instructions + 1 funnel shift instead of 9 + 1,
// with bit-identical keys.
template <int R, int BLOCK, bool COMMON = false>
struct Culler {
    float hx[R], hy[R], hz[R];     // cull direction / sqrt 2: d * sqrt((1 + eps) / 2) / |d|
    float mx[R], my[R], mz[R];     // -2 o
    float P[R];                    // o . h  (with that h)
    float Q[R];                    // |o|^2 (1 - 54 u)
    float cox, coy, coz;           // COMMON: the origin every ray of the kernel's common-origin region starts at

    static constexpr int LIST_WORDS = CHUNK_GROUPS * R;                         // per thread
    static constexpr size_t LIST_BYTES = (size_t)LIST_WORDS * BLOCK * sizeof(uint32_t);   // per CTA

    __device__ __forceinline__ void set_ray(int r, float o_x, float o_y, float o_z, float d_x, float d_y, float d_z) {
        float a = fmaf(d_z, d_z, fmaf(d_y, d_y, d_x * d_x));
        float s = rsqrtf(a) * ((1.0f + 0.5f * CULL_EPS) * 0.70710678118654752f);   // h / sqrt 2, see key_bits
        hx[r] = d_x * s; hy[r] = d_y * s; hz[r] = d_z * s;
        mx[r] = -2.0f * o_x; my[r] = -2.0f * o_y; mz[r] = -2.0f * o_z;
        P[r] = fmaf(o_z, hz[r], fmaf(o_y, hy[r], o_x * hx[r]));
        Q[r] = fmaf(o_z, o_z, fmaf(o_y, o_y, o_x * o_x)) * RAY_DEFLATE;
    }
    // a dead slot.  General form: nc = s - inf = -inf for every sphere, so the key's sign bit is always set.
    // (Common-origin form: nothing about the ray can kill it — the sinks drop a dead ray's words instead.)
    __device__ __forceinline__ void kill(int r) {
        hx[r] = 1.f; hy[r] = 0.f; hz[r] = 0.f;
        mx[r] = my[r] = mz[r] = 0.f;
        P[r] = 0.f;
        Q[r] = CUDART_INF_F;
    }

    // opaque to the optimiser: otherwise ptxas rematerialises h (RSQ + 4 FMUL) per sphere to save registers
    __device__ __forceinline__ void pin() {
        if (COMMON) {
            RT_FOR_R asm volatile("" : "+f"(hx[r]), "+f"(hy[r]), "+f"(hz[r]), "+f"(P[r]));
        } else {
            RT_FOR_R asm volatile("" : "+f"(hx[r]), "+f"(hy[r]), "+f"(hz[r]), "+f"(mx[r]), "+f"(my[r]), "+f"(mz[r]), "+f"(P[r]), "+f"(Q[r]));
        }
    }

    static __device__ __forceinline__ unsigned list_begin(const uint32_t* list) {
        return (unsigned)__cvta_generic_to_shared(list + threadIdx.x);
    }
    static __device__ __forceinline__ unsigned word(const uint32_t* list, int g, int r) {
        return list[(g * R + r) * BLOCK + threadIdx.x];
    }

    // the record of a sphere for rays that all start at o: (-cx, -cy, -cz, (W + 2 o.c) - |o|^2 (1 - 54 u)) — the
    // very operations key_bits applies per ray in the general form, applied once
    static __device__ __forceinline__ float4 common_record(float4 S, float o_x, float o_y, float o_z) {
        const float m_x = -2.0f * o_x, m_y = -2.0f * o_y, m_z = -2.0f * o_z;
        const float q = fmaf(o_z, o_z, fmaf(o_y, o_y, o_x * o_x)) * RAY_DEFLATE;
        S.w = fmaf(S.x, m_x, fmaf(S.y, m_y, fmaf(S.z, m_z, S.w))) - q;
        return S;
    }

    // S = (-cx, -cy, -cz, W = r2i - c.c)   [COMMON: the 4th component is common_record's]
    // b min(b, 0) is evaluated as c c - c |c| with c = b / sqrt 2 (the ray's h and P carry the 1 / sqrt 2): two FFMAs,
    // the second with SASS operand modifiers (-c, |c|), instead of FMNMX + FFMA — the ALU pipe then only sees the
    // funnel shift (loopbench: 11.5 vs 12.1 issue cycles per warp-test)
    __device__ __forceinline__ unsigned key_bits(const float4 S, int r) const {
        float c = fmaf(S.x, hx[r], fmaf(S.y, hy[r], fmaf(S.z, hz[r], P[r])));
        if (COMMON) return __float_as_uint(fmaf(-c, fabsf(c), fmaf(c, c, S.w)));
        float s = fmaf(S.x, mx[r], fmaf(S.y, my[r], fmaf(S.z, mz[r], S.w)));
        return __float_as_uint(fmaf(-c, fabsf(c), fmaf(c, c, s - Q[r])));
    }

    // One chunk: `count` records (a multiple of CULL_PAD, <= CHUNK) starting at shared address sa.  Writes the
    // chunk's mask words and returns the bitmap of the words that hold a survivor: bit 16 r + g = (ray r, group g),
    // so the sinks visit exactly those words (walking every word of a flagged group cost ~30 % of the warps' time).
    __device__ __forceinline__ unsigned long long cull_chunk(unsigned sa, int count, uint32_t* list) const {
        unsigned la = list_begin(list);
        unsigned nzr[R];
        RT_FOR_R nzr[r] = 0u;
        const int full = count / GROUP;
        for (int g = 0; g < full; ++g, la += R * BLOCK * 4) {
            unsigned acc[R];
            RT_FOR_R acc[r] = 0u;                  // all 32 bits are shifted out below
#pragma unroll 8
            for (int u = 0; u < GROUP; ++u, sa += 16) {
                const float4 S = lds128(sa);
                RT_FOR_R acc[r] = __funnelshift_l(key_bits(S, r), acc[r], 1);
            }
            RT_FOR_R {
                asm volatile("st.shared.u32 [%0], %1;" ::"r"(la + (unsigned)(r * BLOCK * 4)), "r"(acc[r]) : "memory");
                nzr[r] |= (acc[r] != 0xffffffffu ? 1u : 0u) << g;
            }
        }
        const int rem = count - full * GROUP;
        if (rem) {                                 // last, partial group of the chunk
            unsigned acc[R];
            RT_FOR_R acc[r] = 0xffffffffu;
            for (int u = 0; u < rem; u += CULL_PAD) {
#pragma unroll
                for (int v = 0; v < CULL_PAD; ++v, sa += 16) {
                    const float4 S = lds128(sa);
                    RT_FOR_R acc[r] = __funnelshift_l(key_bits(S, r), acc[r], 1);
                }
            }
            RT_FOR_R {
                asm volatile("st.shared.u32 [%0], %1;" ::"r"(la + (unsigned)(r * BLOCK * 4)), "r"(acc[r]) : "memory");
                nzr[r] |= (acc[r] != 0xffffffffu ? 1u : 0u) << full;
            }
        }
        unsigned long long nz = 0ull;
        RT_FOR_R nz |= (unsigned long long)nzr[r] << (16 * r);
        return nz;
    }

    // Records [s0, s1) of the resident tile (s1 - s0 a multiple of CULL_PAD), chunk by chunk; kbase = cull index
    // of tile record 0.  Every lane of the warp must call it (sinks use warp collectives).
    template <class Sink>
    __device__ __forceinline__ void run_range(const float4* s_cull, int s0, int s1, int kbase, uint32_t* list, Sink& sink) {
        for (int c0 = s0; c0 < s1; c0 += CHUNK) {
            const int cc = min(CHUNK, s1 - c0);
            const unsigned long long nz = cull_chunk(smem_addr(s_cull + c0), cc, list);
            sink.flush(list, nz, cc, kbase + c0);
        }
    }

    // Whole cull list.  In tiled mode every thread of the CTA must call it (tile loads use __syncthreads).
    // A preloaded scene is a single resident tile s_cull[0, n_cull); a tiled scene streams tiles of `cap` records.
    // Moving spheres are culled as the static bounding sphere of their swept volume (the FP64 refine
    // evaluates the exact moving sphere), so there is ONE hot loop.
    template <class Sink>
    __device__ __forceinline__ void run(const DevScene& sc, float4* s_cull, int cap, bool preloaded, uint32_t* list,
                                        Sink& sink) {
        pin();
        for (int base = 0; base < sc.n_cull; base += cap) {
            const int count = min(cap, sc.n_cull - base);
            if (!preloaded) {
                __syncthreads();
                for (int i = threadIdx.x; i < count; i += BLOCK) {
                    float4 S = __ldg(&sc.cull_a[base + i]);
                    if (COMMON) S = common_record(S, cox, coy, coz);
                    s_cull[i] = S;
                }
                __syncthreads();
            }
            run_range(s_cull, 0, count, base, list, sink);
        }
    }

    // Preloaded scene only: this warp tests slice `part` of `parts` of the sphere groups (a short queue is
    // spread over more warps by splitting the list; PairSink merges the results).
    template <class Sink>
    __device__ __forceinline__ void run_slice(const DevScene& sc, float4* s_cull, uint32_t* list, Sink& sink, int part,
                                              int parts) {
        pin();
        const int groups = (sc.n_cull + GROUP - 1) / GROUP;
        const int s0 = slice_lo(groups, part, parts) * GROUP, s1 = min(slice_lo(groups, part + 1, parts) * GROUP, sc.n_cull);
        run_range(s_cull, s0, s1, 0, list, sink);
    }
};

__device__ __forceinline__ void preload_scene(const DevScene& sc, float4* s_cull, int block) {
    for (int i = threadIdx.x; i < sc.n_cull; i += block) s_cull[i] = __ldg(&sc.cull_a[i]);
    __syncthreads();
}

// Walks the survivors recorded in a thread's mask words: for (it.begin(nz, count); it.next(list, r, k);) ...
// yields (ray r, chunk-relative sphere k) one pair at a time, so a warp runs max-over-lanes(#pairs) iterations.
template <int R, int BLOCK>
struct SurvivorIter {
    unsigned long long z;
    unsigned sv;
    int g, r, m, full, rem;
    __device__ __forceinline__ void begin(unsigned long long nz, int count) {
        z = nz; sv = 0u; g = 0; r = 0; m = 0;
        full = count / GROUP; rem = count - full * GROUP;
    }
    __device__ __forceinline__ bool next(const uint32_t* list, int& ray, int& k) {
        if (sv == 0u) {                      // every flagged word holds at least one survivor
            if (z == 0ull) return false;
            const int i = __ffsll((long long)z) - 1;
            z &= z - 1ull;
            r = i >> 4;
            g = i & 15;
            m = g < full ? GROUP : rem;
            sv = ~Culler<R, BLOCK>::word(list, g, r);
        }
        const int bit = __ffs(sv) - 1;
        sv &= sv - 1u;
        ray = r;
        k = g * GROUP + (m - 1 - bit);
        return true;
    }
};

// ------------------------------------------------------------------------------------------
// RefineSink: the owning thread refines its survivors in FP64 and keeps the closest hit in
// registers (trace kernel, megakernel).  It owns the rays as given (origin, un-normalised
// direction, time); the Culler only holds what the FP32 test needs.
// ------------------------------------------------------------------------------------------
template <int R, int BLOCK, bool GEN = false>
struct RefineSink {
    float ox[R], oy[R], oz[R];     // origin
    float dx[R], dy[R], dz[R];     // direction as given (un-normalised, util.clj:13-16)
    float tm[R];                   // ray time
    double best_t[R];
    int best_k[R];
    unsigned best_tie[R];          // DevScene::tie_hi of the running winner
    unsigned ncand;
    double tmin, tmax;
    const DevScene* sc;
    // path context of the rays (megakernel): what a ConstantMedium needs for its `rand`; has_ctx = false in rt_trace_primary
    bool has_ctx;
    uint2 key;
    uint32_t pix[R], smp[R], bounce[R];

    __device__ __forceinline__ void begin() {
        RT_FOR_R {
            best_t[r] = CUDART_INF;
            best_k[r] = -1;
            best_tie[r] = 0xffffffffu;
        }
    }

    // exact test of (ray r, leaf k): closest t wins, exact ties by DevScene::tie_hi (hitable.clj:17-26 / :99-105)
    __device__ __forceinline__ void refine(int r, int k) {
        float sox = ox[0], soy = oy[0], soz = oz[0], sdx = dx[0], sdy = dy[0], sdz = dz[0], stm = tm[0];
        uint32_t spix = 0, ssmp = 0, sb = 0;
        if (has_ctx) { spix = pix[0]; ssmp = smp[0]; sb = bounce[0]; }
#pragma unroll
        for (int q = 1; q < R; ++q)
            if (r == q) {
                sox = ox[q]; soy = oy[q]; soz = oz[q]; sdx = dx[q]; sdy = dy[q]; sdz = dz[q]; stm = tm[q];
                if (has_ctx) { spix = pix[q]; ssmp = smp[q]; sb = bounce[q]; }
            }
        const double t = refine_leaf<GEN>(sc, k, sox, soy, soz, sdx, sdy, sdz, stm, tmin, tmax, has_ctx, key, spix, ssmp, sb);
        ncand++;
        if (t < CUDART_INF) {
            const unsigned tie = __ldg(&sc->tie_hi[k]);
#pragma unroll
            for (int q = 0; q < R; ++q)
                if (r == q && (t < best_t[q] || (t == best_t[q] && tie < best_tie[q]))) {
                    best_t[q] = t;
                    best_k[q] = k;
                    best_tie[q] = tie;
                }
        }
    }

    __device__ __forceinline__ void flush(const uint32_t* list, unsigned long long nz, int count, int kbase) {
        SurvivorIter<R, BLOCK> it;
        it.begin(nz, count);
        int r, k;
        while (it.next(list, r, k)) refine(r, kbase + k);
    }

    // the spheres that bypass the cull (DevScene::n_list .. n): tested directly for the rays in `live` (bit r)
    __device__ __forceinline__ unsigned direct(unsigned live) {
        unsigned nd = 0;
        for (int k = sc->n_list; k < sc->n; ++k)
            for (int r = 0; r < R; ++r)
                if ((live >> r) & 1u) { refine(r, k); ++nd; }
        ncand -= nd;
        return nd;
    }
};

// ------------------------------------------------------------------------------------------
// Wavefront path tracer: one global queue of paths, one kernel per stage, each at its own occupancy.
//
//   queue record (3 x float4 per path, AoS so one thread moves a path with 3 LDG/STG.128):
//       a = (ox, oy, oz, time)   b = (dx, dy, dz, pixel index)   c = (atten r, g, b, sample << 8 | depth)
//   per bounce ("iteration"), in stream order, all counts on the device:
//     wf_cull      persistent, 2 CTAs/SM: warps claim batches of 32*R queue entries (one atomic per
//                  batch) and run the FP32 brute-force loop with the sphere list in shared memory; the
//                  survivors are only EMITTED as (entry, sphere) pairs — per-lane counts are prefix-
//                  summed with shuffles, one global atomic per warp flush claims the span.  No FP64, no
//                  shading state: this kernel is the hot loop and nothing else.  A short queue switches
//                  to 1 ray per thread and splits the sphere list across warps (the pairs merge later).
//     wf_refine    one thread per pair: FP64 refine with the reference's exact formula, closest t per
//                  entry merged with a 64-bit atomicMin on the double's bit pattern; pairs that were the
//                  running minimum go to a compact candidate list
//     wf_tiebreak  candidates owning the final minimum t race with atomicMin on (caller index, k): exact
//                  ties go to the lower caller index, the Hitlist rule (hitable.clj:17-26)
//                  (a single 128-bit CAS merge was tried and was 2.4x slower than this two-step)
//     wf_shade     one thread per entry: scatter / emitted, accumulate, then compact: surviving paths
//                  and fresh camera rays for finished lanes are appended to the next queue (warp ballot
//                  + prefix popc + one atomic per warp, same for the (sample, pixel) work counter)
//   The host enqueues iterations ahead and polls the queue count every few iterations.
// ------------------------------------------------------------------------------------------
// A queue holds two populations: paths in flight at [0, cnt[q][0]) and FRESH camera rays at [capacity - cnt[q][1],
// capacity).  A fresh entry is only a promise: entry capacity - cnt[q][1] + i stands for work item gen_base[q] + i, and
// the cull kernel GENERATES its ray (get-ray, camera.clj:35-48) when it first needs it, and writes the queue record for the
// later stages.  When every camera ray starts at the same origin (WaveParams::base.common_origin) the cull runs its
// common-origin form over the fresh region (Culler<.., COMMON>).  The last CTA of wf_shade hands out the next
// iteration's fresh work: ONE atomic on the shared (sample, pixel) counter per launch.
struct alignas(8) WaveState {
    unsigned cnt[2][2];
    unsigned long long gen_base[2];
    unsigned batch;                // next batch (wf_cull)
    unsigned npairs;               // pairs emitted this iteration
    unsigned exhausted;            // the (sample, pixel) work counter has run past the end
    unsigned done;                 // CTAs of the running wf_shade launch that have finished (the last one takes the ticket)
    unsigned mode;                 // MODE_RUN, or MODE_DONE once the lane has drained (set on the device by the last CTA of
                                   // wf_shade / wf_tail): kernels queued past the end look at it and return at once
    unsigned pad;                  // PAIR_NULL padding slots among this iteration's npairs (wf_cull_tc reserves pair slots in chunks)
};
enum { MODE_RUN = 0, MODE_DONE = 2 };
// What the host needs to know about a lane, written by the device straight into pinned, mapped HOST memory by the last
// CTA of every wf_shade (and of wf_tail): no copy, no event, nothing in the lane's stream.  `seq` is written last.
struct LaneStatus {
    unsigned n_next;               // entries the next iteration will find (paths in flight + fresh)
    unsigned n_fresh;              // of which fresh
    unsigned exhausted;            // the (sample, pixel) counter has run out: the population only shrinks from here
    unsigned mode;
    unsigned seq;                  // iterations of this render completed on the device
    unsigned pad[3];
};
// entry index of the i-th entry of a queue holding n_g general and n_p common-origin entries
__device__ __forceinline__ unsigned wf_entry(unsigned i, unsigned n_g, unsigned n_p, unsigned capacity) {
    return i < n_g ? i : capacity - n_p + (i - n_g);
}

// Timeline tracing (RT_TRACE=<file>): every wavefront kernel launch owns one record; thread 0 of every CTA folds its
// entry / exit %globaltimer into it.  Shows how the two lanes' kernels really interleave on the device (ncu serialises
// them; there is no nsys in this environment).
struct TraceRec {
    unsigned long long t_start, t_end;   // ns, %globaltimer; min over CTAs / max over CTAs
};
__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
struct TraceScope {
    TraceRec* rec;
    __device__ __forceinline__ explicit TraceScope(TraceRec* r) : rec(r) {
        if (rec && threadIdx.x == 0) atomicMin(&rec->t_start, global_timer_ns());
    }
    __device__ __forceinline__ ~TraceScope() {
        if (rec && threadIdx.x == 0) atomicMax(&rec->t_end, global_timer_ns());
    }
};

struct WaveParams {
    RenderParams base;
    float4* queue[2];              // 3 * capacity float4 each
    unsigned long long* best_t;    // [capacity] closest t (double bits)
    unsigned long long* best_key;  // [capacity] (caller index + 1) << 32 | k
    uint2* pairs;                  // [pair_cap] (entry, k)
    uint2* cands;                  // [pair_cap] pairs that were the running minimum when they merged
    double* cand_t;                // [pair_cap + slack] their t
    unsigned* cand_count;          // [warps of the refine grid] candidates in each warp's private region
    WaveState* st;
    int capacity;                  // multiple of 32
    unsigned pair_cap;
    int cur;                       // queue read by this iteration
    int claims_per_warp;           // wf_cull: 0 = persistent warps (claim batches until none is left); k > 0 = a warp retires
                                   // after k batches (many short CTAs: the SM's slots turn over, so the other lane's
                                   // high-priority stage kernels get on the SM while this cull is still running)
    int resident_warps;            // wf_cull warps resident on the device at once (sizes the balancing tail); 0 = the grid's
    volatile LaneStatus* status;   // the lane's status record in mapped host memory (null inside wf_tail's per-CTA views)
    unsigned iter;                 // 1-based number of this iteration within the render (LaneStatus::seq after its wf_shade)
    TraceRec* trace;               // this launch's timeline record, or null
    int tc_slots;                  // wf_cull_tc: ray-tile buffers in shared memory (2 .. 4)
    int tc_tile0, tc_launch_tiles; // wf_cull_tc: this launch tests feature tiles [tc_tile0, tc_tile0 + tc_launch_tiles) of the list (<= 4: they
    int tc_pass;                   //   stay resident in shared memory); a longer list takes several launches ("passes") per iteration, and only
                                   //   pass 0 generates the fresh entries' rays and counts the rays
    unsigned tail_solo;            // wf_tail: a slice that has shrunk to this many paths or fewer is finished by groups of tail_lpp lanes,
    unsigned tail_lpp;             //   each running one path at a time to its end (wf_solo_paths); tail_lpp = 8 | 16 | 32
};
__device__ __forceinline__ void publish_status(const WaveParams& W, unsigned n_next, unsigned n_fresh, unsigned exhausted, unsigned mode,
                                               unsigned seq) {
    if (!W.status) return;
    W.status->n_next = n_next;
    W.status->n_fresh = n_fresh;
    W.status->exhausted = exhausted;
    W.status->mode = mode;
    __threadfence_system();
    W.status->seq = seq;
}

constexpr unsigned long long BEST_T_INIT = 0x7ff0000000000000ull;   // +inf
constexpr unsigned long long BEST_KEY_MISS = ~0ull;
constexpr unsigned long long BEST_KEY_OVERFLOW = 0ull;              // survives every atomicMin
constexpr unsigned PAIR_NULL = 0xffffffffu;

// claim consecutive slots for the lanes whose predicate is set (one atomic per warp); returns this lane's slot
__device__ __forceinline__ unsigned warp_claim(unsigned* counter, bool pred, unsigned lane) {
    unsigned m = __ballot_sync(0xffffffffu, pred);
    unsigned base = 0;
    if (m) {
        int leader = __ffs(m) - 1;
        if ((int)lane == leader) base = atomicAdd(counter, (unsigned)__popc(m));
        base = __shfl_sync(0xffffffffu, base, leader);
    }
    return base + __popc(m & ((1u << lane) - 1u));
}

// rt_render_views: camera ray of view v's pixel (i, j) (view-local), out of line so that the single-camera path of the
// kernels that generate rays keeps its registers
struct CameraRay {
    float3 o, d;
    float time;
};
__device__ __noinline__ CameraRay view_ray(const DevCamera* __restrict__ views, uint32_t v, int nx, int ny, int i, int j,
                                           uint32_t pixel, uint32_t sample, uint2 key) {
    CameraRay r;
    generate_ray(views[v], nx, ny, i, j, pixel, sample, key, r.o, r.d, r.time, nullptr);
    return r;
}

// camera ray of work item w as a queue record.  VIEWS = false: a kernel instantiated for single-camera renders only.
template <bool VIEWS>
__device__ __forceinline__ void make_path(const RenderParams& P, unsigned long long w, float4& a, float4& b, float4& c) {
    const unsigned pshard = (unsigned)P.nx * (unsigned)P.rows_in_shard;
    unsigned s_local, q;
    if (P.total_work <= 0xffffffffull) {     // warp-uniform: a 32-bit divide is ~4x fewer instructions than the 64-bit one
        s_local = (unsigned)w / pshard;
        q = (unsigned)w - s_local * pshard;
    } else {
        s_local = (unsigned)(w / pshard);
        q = (unsigned)(w - (unsigned long long)s_local * pshard);
    }
    int row_local = (int)(q / (unsigned)P.nx);
    int i = (int)(q - (unsigned)row_local * (unsigned)P.nx);
    int j = P.row_offset + row_local * P.row_stride;
    uint32_t pix = (uint32_t)j * (uint32_t)P.nx + (uint32_t)i;
    uint32_t smp = (uint32_t)(P.sample_begin + (int)s_local);
    uint32_t slot = pix;
    if (P.path_pixel) {                       // rt_trace_paths: work item w is path w of the caller's list
        pix = (uint32_t)__ldg(&P.path_pixel[w]);
        smp = (uint32_t)__ldg(&P.path_sample[w]);
        j = (int)(pix / (uint32_t)P.nx);
        i = (int)(pix - (uint32_t)j * (uint32_t)P.nx);
        slot = (uint32_t)w;
    }
    float3 o, d;
    float tmv;
    if (VIEWS && P.views && !P.path_pixel) {  // rt_render_views: the view's camera, view-local row and Philox pixel
        const uint32_t v = view_of(P, slot);
        pix = slot - v * P.view_px;
        slot = pix | (v << P.view_bits);
        const CameraRay r = view_ray(P.views, v, P.nx, P.ny, i, j - (int)v * P.ny, pix, smp, P.key);
        o = r.o; d = r.d; tmv = r.time;
    } else {
        generate_ray(P.cam, P.nx, P.ny, i, j, pix, smp, P.key, o, d, tmv, nullptr);
    }
    a = make_float4(o.x, o.y, o.z, tmv);
    b = make_float4(d.x, d.y, d.z, __uint_as_float(slot));
    c = make_float4(1.f, 1.f, 1.f, __uint_as_float((smp << 8) | (uint32_t)P.max_depth));
}

// Start of a render: every lane's queue 0 holds only fresh entries (work items [first, first + count) of the lane), the
// shared work counter starts past every lane's first fill.  No ray is generated here: the first cull does that.
constexpr int kMaxLanes = 2;
struct InitParams {
    WaveState* st[kMaxLanes];
    unsigned long long first[kMaxLanes];
    unsigned count[kMaxLanes];
    int n_lanes;
    unsigned long long* work_counter;
    unsigned long long* counters;
    unsigned long long total0, total_work;
};
__global__ void wf_init(const InitParams I) {
    for (int l = 0; l < I.n_lanes; ++l) {
        WaveState* st = I.st[l];
        st->cnt[0][0] = 0; st->cnt[0][1] = I.count[l];
        st->cnt[1][0] = 0; st->cnt[1][1] = 0;
        st->gen_base[0] = I.first[l]; st->gen_base[1] = 0;
        st->batch = 0; st->npairs = 0; st->done = 0; st->mode = I.count[l] ? MODE_RUN : MODE_DONE; st->pad = 0;
        st->exhausted = I.total0 >= I.total_work ? 1u : 0u;
    }
    *I.work_counter = I.total0;
    atomicAdd(&I.counters[DC_SAMPLES], I.total0);
}
// closest-hit words of a lane -> (+inf, MISS).  wf_shade leaves them that way (the consumer of an entry's words resets
// them), so this runs only after an allocation or after a render that did not run to completion.
__global__ void wf_fill_best(unsigned long long* best_t, unsigned long long* best_key, size_t n) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        best_t[i] = 0x7ff0000000000000ull;
        best_key[i] = ~0ull;
    }
}

// PairSink: survivors leave the cull kernel as (entry, sphere) pairs.  Called warp-converged: per-lane
// pair counts are prefix-summed with shuffles and ONE global atomic claims the warp's span.
// A warp whose span does not fit marks its entries OVERFLOW; wf_shade re-intersects those exactly.
template <int R, int BLOCK>
struct PairSink {
    unsigned idx0;                 // VIRTUAL index of ray r = idx0 + 32 r; queue entry = entry(idx0 + 32 r)
    unsigned n;                    // end of the virtual range being culled
    unsigned n_g, p0;              // virtual index v < n_g is entry v, else entry p0 + (v - n_g) (n_g = ~0: identity)
    __device__ __forceinline__ unsigned entry(unsigned v) const { return v < n_g ? v : p0 + (v - n_g); }
    unsigned long long live;       // bits 16 r .. 16 r + 15 set if ray r of this lane is a live entry
    uint2* pairs;                  // by value (not a WaveParams*): keeps a caller's modified copy of the params in registers
    unsigned pair_cap;
    unsigned long long* best_key;
    WaveState* st;

    __device__ __forceinline__ void flush(const uint32_t* list, unsigned long long nz, int count, int kbase) {
        nz &= live;                                    // a dead ray's words (common-origin form) are not survivors
        if (!__any_sync(0xffffffffu, nz != 0ull)) return;
        const unsigned lane = threadIdx.x & 31u;
        unsigned np = 0;
        for (unsigned long long z = nz; z; z &= z - 1ull) {
            const int i = __ffsll((long long)z) - 1;
            np += __popc(~Culler<R, BLOCK>::word(list, i & 15, i >> 4));
        }
        unsigned incl = np;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            unsigned v = __shfl_up_sync(0xffffffffu, incl, d);
            if ((int)lane >= d) incl += v;
        }
        const unsigned total = __shfl_sync(0xffffffffu, incl, 31);
        unsigned base = 0;
        if (lane == 0) base = atomicAdd(&st->npairs, total);
        base = __shfl_sync(0xffffffffu, base, 0);
        const bool fits = base + total <= pair_cap;
        unsigned w = base + incl - np;
        SurvivorIter<R, BLOCK> it;
        it.begin(nz, count);
        int r, k;
        while (it.next(list, r, k)) {
            const unsigned v = idx0 + 32u * (unsigned)r;
            if (fits) {
                pairs[w] = make_uint2(entry(v), (unsigned)(kbase + k));
            } else {
                if (w < pair_cap) pairs[w] = make_uint2(PAIR_NULL, 0u);
                if (v < n) best_key[entry(v)] = BEST_KEY_OVERFLOW;   // nothing else writes the word during the cull
            }
            ++w;
        }
    }
};

// Virtual entries [e0, e1) in batches of 32*R, each batch optionally split into `parts` sphere slices.  Virtual index
// v < n_g is queue entry v (a path in flight: its ray is loaded); v >= n_g is entry p0 + (v - n_g), FRESH: the ray of
// work item gen0 + (v - n_g) is generated here and its queue record written for the later stages.  The
// (batch, slice) work items of this range are numbered item0, item0 + 1, ...; warps claim item numbers from the
// shared counter (preloaded scenes) or take them in a CTA-uniform static order (tiled scenes).  `claimed` is an
// item number this warp has already claimed (or ~0u); returns the first claimed number beyond the range, so a
// following range can use it.
constexpr unsigned ITEM_NONE = 0xffffffffu;
constexpr unsigned ITEM_STOP = 0xfffffffeu;   // this warp has used up its claims (WaveParams::claims_per_warp)
// The CTAs that cooperate on one queue: the whole grid (bid = blockIdx.x of nblk = gridDim.x), or a single CTA
// working alone on its own slice of the queue (bid 0 of 1; wf_tail).
struct Scope {
    unsigned bid, nblk;
};
__device__ __forceinline__ Scope grid_scope() { return Scope{blockIdx.x, gridDim.x}; }
template <int R, int BLOCK, bool COMMON, bool VIEWS>
__device__ __forceinline__ unsigned wf_cull_batches(const WaveParams& W, Scope sc_, int cur, unsigned e0, unsigned e1, unsigned n_g,
                                                    unsigned p0, unsigned long long gen0, int parts, unsigned item0, unsigned claimed,
                                                    int& budget, float4* s_cull, uint32_t* s_list) {
    if (claimed == ITEM_STOP) return ITEM_STOP;
    const RenderParams& P = W.base;
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, warps = BLOCK / 32;
    const unsigned n_batches = (e1 - e0 + 32 * R - 1) / (32 * R);
    const unsigned n_items = n_batches * (unsigned)parts;          // (batch, sphere slice) work items
    Culler<R, BLOCK, COMMON> K;
    K.cox = P.cam.origin.x; K.coy = P.cam.origin.y; K.coz = P.cam.origin.z;
    PairSink<R, BLOCK> sink;
    sink.n = e1;
    sink.n_g = n_g;
    sink.p0 = p0;
    sink.pairs = W.pairs;
    sink.pair_cap = W.pair_cap;
    sink.best_key = W.best_key;
    sink.st = W.st;
    unsigned item = sc_.bid * warps + warp;                        // tiled scenes: CTA-uniform static order
    const unsigned uniform_end = (n_items + warps - 1) / warps * warps;
    for (;;) {
        if (P.preloaded) {
            if (claimed != ITEM_NONE) {
                item = claimed;
                claimed = ITEM_NONE;
            } else {
                unsigned b = 0;
                if (lane == 0) b = atomicAdd(&W.st->batch, 1u);
                item = __shfl_sync(0xffffffffu, b, 0);
            }
            if (item >= item0 + n_items) return item;
            item -= item0;
        } else {
            if (item - warp >= uniform_end) break;
        }
        const unsigned batch = item / (unsigned)parts, part = item - batch * (unsigned)parts;
        sink.idx0 = e0 + batch * (32 * R) + lane;     // ray r of this lane = entry idx0 + 32 r
        sink.live = 0ull;
        RT_FOR_R {
            const unsigned v = sink.idx0 + 32 * r;
            if (v < e1 && batch < n_batches) {
                float4* qc = cur ? W.queue[1] : W.queue[0];   // a select, not a dynamic index (keeps copies of W in registers)
                float4 a, b;
                if (v >= n_g) {                               // fresh: generate the camera ray of its work item
                    float4 c;
                    float4* q = qc + 3 * (size_t)(p0 + (v - n_g));
                    make_path<VIEWS>(P, gen0 + (v - n_g), a, b, c);
                    if (part == 0) { q[0] = a; q[1] = b; q[2] = c; }
                } else {
                    a = qc[3 * (size_t)v];
                    b = qc[3 * (size_t)v + 1];
                }
                K.set_ray(r, a.x, a.y, a.z, b.x, b.y, b.z);
                sink.live |= 0xffffull << (16 * r);
            } else {
                K.kill(r);
            }
        }
        if (parts > 1) K.run_slice(P.sc, s_cull, s_list, sink, (int)part, parts);
        else           K.run(P.sc, s_cull, P.cull_cap, P.preloaded != 0, s_list, sink);
        item += sc_.nblk * warps;
        if (P.preloaded && budget > 0 && --budget == 0) return ITEM_STOP;
    }
    return ITEM_NONE;
}

// The shape of the cull work.  The queue holds n_p fresh entries (camera rays, generated here; when they all share an
// origin they are culled in the cheaper common-origin form against the tile s_cullc) and n_g paths in flight.  A long
// queue: batches of R rays per thread for the bulk of both, then — so that the warps do not finish up to a whole 32*R
// batch apart — one-ray batches for the last stretch (two per warp of the grid), all claimed from the same counter.  A
// short queue: 1 ray per thread, and below two batches per warp the sphere list is split across warps too (the pairs
// merge in wf_refine).  R = 1 instantiates only the short form.  s_cullc may be null when n_p is 0 (the tail).
template <int R, int BLOCK, bool VIEWS>
__device__ __forceinline__ void wf_cull_body(const WaveParams& W, Scope sc_, int cur, unsigned n_g, unsigned n_p, unsigned long long gen_base,
                                             float4* s_cull, float4* s_cullc, uint32_t* s_list) {
    const RenderParams& P = W.base;
    const unsigned n = n_g + n_p, p0 = (unsigned)W.capacity - n_p;
    if (sc_.bid == 0 && threadIdx.x == 0) atomicAdd(&P.counters[DC_RAYS], (unsigned long long)n);
    const unsigned grid_warps = W.resident_warps > 0 ? (unsigned)W.resident_warps : sc_.nblk * (BLOCK / 32);
    int budget = W.claims_per_warp;
    // two virtual ranges: C = the fresh entries in the common-origin form (identity mapping over [p0, p0 + n_c)), and
    // V = everything culled in the general form: the n_g paths in flight, followed — when the camera rays do NOT share an
    // origin (a real aperture) — by the fresh entries (virtual index >= n_g)
    const unsigned n_c = P.common_origin ? n_p : 0u, n_v = n - n_c;
    const unsigned long long genC = gen_base - p0;   // C: virtual index = entry index; item = gen_base + (entry - p0)
    if (R > 1 && !P.preloaded) {
        // tiled scene: CTA-uniform static order; the tile loader builds the common-origin records itself
        if (n_c) wf_cull_batches<R, BLOCK, true, VIEWS>(W, sc_, cur, p0, p0 + n_c, 0u, 0u, genC + 0u, 1, 0u, ITEM_NONE, budget, s_cull, s_list);
        if (n_v) wf_cull_batches<R, BLOCK, false, VIEWS>(W, sc_, cur, 0u, n_v, n_g, p0, gen_base, 1, 0u, ITEM_NONE, budget, s_cull, s_list);
    } else if (R > 1 && n >= grid_warps * 64u) {
        const unsigned tail = grid_warps * 64u, per = 32u * R;                       // two one-ray batches per warp
        const unsigned g_rest0 = min(n_v, tail), p_rest0 = min(n_c, tail - g_rest0);
        const unsigned g_bulk = (n_v - g_rest0) / per * per, p_bulk = (n_c - p_rest0) / per * per;
        unsigned items = 0;
        unsigned next = wf_cull_batches<R, BLOCK, true, VIEWS>(W, sc_, cur, p0, p0 + p_bulk, 0u, 0u, genC, 1, items, ITEM_NONE, budget, s_cullc, s_list);
        items += p_bulk / per;
        next = wf_cull_batches<R, BLOCK, false, VIEWS>(W, sc_, cur, 0u, g_bulk, n_g, p0, gen_base, 1, items, next, budget, s_cull, s_list);
        items += g_bulk / per;
        next = wf_cull_batches<1, BLOCK, true, VIEWS>(W, sc_, cur, p0 + p_bulk, p0 + n_c, 0u, 0u, genC, 1, items, next, budget, s_cullc, s_list);
        items += (n_c - p_bulk + 31u) / 32u;
        wf_cull_batches<1, BLOCK, false, VIEWS>(W, sc_, cur, g_bulk, n_v, n_g, p0, gen_base, 1, items, next, budget, s_cull, s_list);
    } else {
        const unsigned b1 = (n + 31) / 32;
        int parts = 1;
        if (P.preloaded)
            while (parts < 16 && b1 * (unsigned)parts * 2u <= grid_warps) parts *= 2;
        unsigned next = ITEM_NONE, items = 0;
        if (n_c) {
            next = wf_cull_batches<1, BLOCK, true, VIEWS>(W, sc_, cur, p0, p0 + n_c, 0u, 0u, genC, parts, 0u, ITEM_NONE, budget, P.preloaded ? s_cullc : s_cull, s_list);
            items = (n_c + 31u) / 32u * (unsigned)parts;
        }
        if (n_v) wf_cull_batches<1, BLOCK, false, VIEWS>(W, sc_, cur, 0u, n_v, n_g, p0, gen_base, parts, items, next, budget, s_cull, s_list);
    }
}

// VIEWS: instantiated for rt_render_views (false: single-camera renders, whose camera rays never leave P.cam)
template <int R, int BLOCK, int MINB, bool VIEWS>
__global__ void __launch_bounds__(BLOCK, MINB) wf_cull(const __grid_constant__ WaveParams W) {
    TraceScope trace(W.trace);
    const RenderParams& P = W.base;
    extern __shared__ float4 smem_f4[];
    float4* s_cull = smem_f4;
    uint32_t* s_list = reinterpret_cast<uint32_t*>(smem_f4 + P.cull_cap);
    float4* s_cullc = reinterpret_cast<float4*>(s_list + Culler<R, BLOCK>::LIST_WORDS * BLOCK);   // common-origin records
    if (W.st->mode != MODE_RUN) return;
    const unsigned n_g = W.st->cnt[W.cur][0], n_p = W.st->cnt[W.cur][1];
    if (n_g + n_p == 0) return;
    const unsigned long long gen_base = W.st->gen_base[W.cur];
    if (P.preloaded) {
        preload_scene(P.sc, s_cull, BLOCK);
        if (n_p && P.common_origin)
            for (int i = threadIdx.x; i < P.sc.n_cull; i += BLOCK)
                s_cullc[i] = Culler<R, BLOCK, true>::common_record(s_cull[i], P.cam.origin.x, P.cam.origin.y, P.cam.origin.z);
    }
    __syncthreads();
    wf_cull_body<R, BLOCK, VIEWS>(W, grid_scope(), W.cur, n_g, n_p, gen_base, s_cull, s_cullc, s_list);
}

#include "rt_cull_tc.cuh"   // wf_cull_tc: the same cull on the tensor cores (tcgen05 / TMEM)

// one thread per pair: FP64 refine + 64-bit atomicMin on the bit pattern of t (> 0, so the order is preserved).
// The atomic's result is NOT consumed (fire-and-forget RED; a returning ATOM made this kernel 3x slower):
// a plain L2 read of the running minimum beforehand decides whether the pair can still be the winner
// (the final winner always passes: the minimum only ever decreases towards its t).  Such pairs are kept
// for the tie-break pass in a region private to the warp — no slot-claim atomics either.
__device__ __forceinline__ unsigned wf_cand_region(const WaveParams& W, unsigned total_warps) {
    return ((W.pair_cap + total_warps * 32u - 1u) / (total_warps * 32u)) * 32u;   // pairs one warp can see
}

// scp: the scene in the kernel's (grid-constant) parameter space — never the address of a local copy of the parameters
template <bool GEN, bool VIEWS>
__device__ __forceinline__ void wf_refine_body(const WaveParams& W, const DevScene* scp, Scope sc_, int cur) {
    const RenderParams& P = W.base;
    const unsigned npairs = min(W.st->npairs, W.pair_cap);
    const unsigned lane = threadIdx.x & 31u;
    if (sc_.bid == 0 && threadIdx.x == 0) {
        W.st->batch = 0;               // wf_cull is done with it
        W.st->cnt[cur ^ 1][0] = 0;     // wf_shade appends to both regions of the other queue next
        W.st->cnt[cur ^ 1][1] = 0;
        atomicAdd(&P.counters[DC_CANDIDATES], (unsigned long long)(npairs - min(npairs, W.st->pad)));   // real pairs (wf_cull_tc pads its reservations); the direct spheres' exact tests are counted apart (DC_DIRECT)
        W.st->pad = 0;
    }
    const unsigned total_warps = sc_.nblk * (blockDim.x >> 5);
    const unsigned warp_id = sc_.bid * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const size_t region = (size_t)warp_id * wf_cand_region(W, total_warps);
    unsigned cnt = 0;
    const unsigned stride = sc_.nblk * blockDim.x;
    // the pair of the NEXT trip is loaded before this trip's pair is refined: its latency hides behind the gathers
    // and the FP64 test of the current one (the loop is a chain of dependent loads: pair -> ray -> sphere)
    const unsigned i_first = sc_.bid * blockDim.x + threadIdx.x;
    uint2 pr_next = i_first < npairs ? W.pairs[i_first] : make_uint2(PAIR_NULL, 0u);
    for (unsigned i0 = i_first - lane; i0 < npairs; i0 += stride) {   // warp-uniform
        const uint2 pr = pr_next;
        const unsigned i_next = i0 + lane + stride;
        pr_next = i_next < npairs ? W.pairs[i_next] : make_uint2(PAIR_NULL, 0u);
        bool cand = false;
        double t = CUDART_INF;
        if (pr.x != PAIR_NULL) {
            const float4* qc = cur ? W.queue[1] : W.queue[0];
            const float4 a = qc[3 * (size_t)pr.x], b = qc[3 * (size_t)pr.x + 1];
            const unsigned long long seen = __ldcg(&W.best_t[pr.x]);
            if (!GEN) {
                t = refine_candidate(P.sc.ex_c0r, P.sc.ex_c1, P.sc.ex_t0t1, P.sc.flags, (int)pr.y, a.x, a.y, a.z, b.x, b.y, b.z,
                                     a.w, 0.001, (double)FLT_MAX);   // core.clj:25 t-range
            } else {
                uint32_t pixq = 0, smpq = 0, bq = 0;
                if (__ldg(&P.sc.prim_type[pr.y]) == PRIM_MEDIUM) {   // its `rand` is keyed by the path (hitable.clj:529)
                    const uint32_t sd = __float_as_uint(qc[3 * (size_t)pr.x + 2].w);
                    pixq = rng_pixel<VIEWS>(P, __float_as_uint(b.w));
                    smpq = sd >> 8;
                    bq = (uint32_t)(P.max_depth - (int)(sd & 255u) + 1);
                }
                t = refine_leaf<true>(scp, (int)pr.y, a.x, a.y, a.z, b.x, b.y, b.z, a.w, 0.001, (double)FLT_MAX, true, P.key, pixq, smpq, bq);
            }
            const unsigned long long tb = (unsigned long long)__double_as_longlong(t);
            if (t < CUDART_INF && tb <= seen) {
                atomicMin(&W.best_t[pr.x], tb);
                cand = true;
            }
        }
        const unsigned m = __ballot_sync(0xffffffffu, cand);
        if (cand) {
            const size_t slot = region + cnt + __popc(m & ((1u << lane) - 1u));
            W.cands[slot] = pr;
            W.cand_t[slot] = t;
        }
        cnt += __popc(m);
    }
    if (lane == 0) W.cand_count[warp_id] = cnt;
}
template <bool GEN, bool VIEWS>
__global__ void __launch_bounds__(256) wf_refine(const __grid_constant__ WaveParams W) {
    if (W.st->mode != MODE_RUN) return;
    TraceScope trace(W.trace);
    wf_refine_body<GEN, VIEWS>(W, &W.base.sc, grid_scope(), W.cur);
}

// exact ties go to the lower caller index, the Hitlist rule (hitable.clj:17-26): candidates that own the final
// minimum t race with atomicMin on (caller index, k).  Same grid shape as wf_refine (warp-private regions).
__device__ __forceinline__ void wf_tiebreak_body(const WaveParams& W, Scope sc_) {
    const RenderParams& P = W.base;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned total_warps = sc_.nblk * (blockDim.x >> 5);
    const unsigned warp_id = sc_.bid * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const size_t region = (size_t)warp_id * wf_cand_region(W, total_warps);
    const unsigned cnt = W.cand_count[warp_id];
    for (unsigned j = lane; j < cnt; j += 32) {
        const uint2 pr = W.cands[region + j];
        if ((unsigned long long)__double_as_longlong(W.cand_t[region + j]) == W.best_t[pr.x])
            atomicMin(&W.best_key[pr.x], (((unsigned long long)__ldg(&P.sc.tie_hi[pr.y])) << 32) | pr.y);
    }
}
__global__ void __launch_bounds__(256) wf_tiebreak(const __grid_constant__ WaveParams W) {
    if (W.st->mode != MODE_RUN) return;
    TraceScope trace(W.trace);
    wf_tiebreak_body(W, grid_scope());
}

// exact closest hit of one ray by brute force in FP64 (only for entries whose pairs overflowed the pair buffer)
template <bool GEN>
__device__ __noinline__ void exact_closest_hit(const DevScene* sc, float ox, float oy, float oz, float dx, float dy, float dz,
                                               float tm, uint2 key, uint32_t pixel, uint32_t sample, uint32_t bounce, double* out_t,
                                               int* out_k) {
    double best = CUDART_INF;
    int bk = -1;
    unsigned btie = 0xffffffffu;
    for (int k = 0; k < sc->n; ++k) {
        double t = refine_leaf<GEN>(sc, k, ox, oy, oz, dx, dy, dz, tm, 0.001, (double)FLT_MAX, true, key, pixel, sample, bounce);
        if (t < CUDART_INF) {
            unsigned tie = __ldg(&sc->tie_hi[k]);
            if (t < best || (t == best && tie < btie)) { best = t; bk = k; btie = tie; }
        }
    }
    *out_t = best;
    *out_k = bk;
}

// s_ctr: shared counters of the calling kernel (DC_COUNT slots, zeroed by the caller); returns samples generated
template <bool GEN, bool VIEWS>
__device__ __forceinline__ unsigned wf_shade_body(const WaveParams& W, const DevScene* scp, Scope sc_, int cur, unsigned* s_ctr) {
    const RenderParams& P = W.base;
    const unsigned n_g = W.st->cnt[cur][0], n_p = W.st->cnt[cur][1], n = n_g + n_p;
    const unsigned lane = threadIdx.x & 31u;
    const float4* qc = cur ? W.queue[1] : W.queue[0];
    float4* qn = cur ? W.queue[0] : W.queue[1];
    if (sc_.bid == 0 && threadIdx.x == 0) W.st->npairs = 0;   // refine / tie-break are done with it
    unsigned n_direct = 0;
    const unsigned stride = sc_.nblk * blockDim.x;
    for (unsigned idx0 = sc_.bid * blockDim.x + threadIdx.x - lane; idx0 < n; idx0 += stride) {   // warp-uniform
        const bool have = idx0 + lane < n;
        const unsigned idx = wf_entry(idx0 + lane, n_g, n_p, (unsigned)W.capacity);
        bool cont = false;
        float4 a, b, c;
        if (have) {
            a = qc[3 * (size_t)idx]; b = qc[3 * (size_t)idx + 1]; c = qc[3 * (size_t)idx + 2];
            unsigned long long key = W.best_key[idx];
            const uint32_t slot = __float_as_uint(b.w), sd = __float_as_uint(c.w);   // slot: the pixel (a render) / the path (rt_trace_paths)
            const uint32_t pix = rng_pixel<VIEWS>(P, slot);
            const uint32_t smp = sd >> 8;
            const int depth = (int)(sd & 255u);
            const uint32_t bounce = (uint32_t)(P.max_depth - depth + 1);
            int k = (int)(unsigned)key;
            double td = __longlong_as_double((long long)W.best_t[idx]);
            // this thread is the last reader of the entry's closest-hit words: it leaves them reset for the next
            // iteration's entry at this index (the cull and the refine only ever lower them; nothing else initialises them)
            W.best_key[idx] = BEST_KEY_MISS;
            W.best_t[idx] = BEST_T_INIT;
            if (key == BEST_KEY_OVERFLOW) {                 // overflow mark: exact brute force for this entry
                exact_closest_hit<GEN>(scp, a.x, a.y, a.z, b.x, b.y, b.z, a.w, P.key, pix, smp, bounce, &td, &k);
                key = k < 0 ? BEST_KEY_MISS : 1ull;
            } else {
                // the spheres that bypass the cull (enclosing spheres: the cull would pass them for nearly every
                // ray) are tested here, exactly, from the registers that hold the ray anyway; same merge rule
                for (int kd = P.sc.n_list; kd < P.sc.n; ++kd) {
                    ++n_direct;
                    const double t = refine_leaf<GEN>(scp, kd, a.x, a.y, a.z, b.x, b.y, b.z, a.w, 0.001, (double)FLT_MAX, true, P.key, pix,
                                                      smp, bounce);   // core.clj:25 t-range
                    const unsigned long long kk = (((unsigned long long)__ldg(&P.sc.tie_hi[kd])) << 32) | (unsigned)kd;
                    if (t < td || (t < CUDART_INF && t == td && kk < key)) {
                        td = t;
                        key = kk;
                        k = kd;
                    }
                }
            }
            const bool hit = key != BEST_KEY_MISS;
            if (P.path_pixel) path_log_ray(P, slot, (int)bounce - 1, a, b, hit ? k : -1, hit ? td : CUDART_INF);
            if (!hit) {                                     // core.clj:40-41 miss -> accum (black)
                atomicAdd(&s_ctr[DC_TERM_MISS], 1u);
                if (P.path_pixel) path_log_end(P, slot, (int)bounce, TERM_MISS);
            } else {
                float3 o = f3(a.x, a.y, a.z), d = f3(b.x, b.y, b.z);
                float3 att, em;
                int reason = TERM_NONE;
                float tmv = a.w;
                ScatterRng rng{P.key, pix, smp, bounce, nullptr, nullptr};
                cont = shade_hit<GEN>(P.sc, scp, k, (float)td, o, d, tmv, depth > 0, rng, att, em, reason);
                if (em.x != 0.f || em.y != 0.f || em.z != 0.f) {   // accum += atten * emitted (core.clj:32-34,37-39)
                    float* dst = P.sum + (size_t)frame_slot<VIEWS>(P, slot) * 3;
                    atomicAdd(dst + 0, c.x * em.x);
                    atomicAdd(dst + 1, c.y * em.y);
                    atomicAdd(dst + 2, c.z * em.z);
                }
                if (cont) {
                    a = make_float4(o.x, o.y, o.z, tmv);
                    b = make_float4(d.x, d.y, d.z, b.w);
                    c = make_float4(c.x * att.x, c.y * att.y, c.z * att.z, __uint_as_float((smp << 8) | (uint32_t)(depth - 1)));
                } else {
                    atomicAdd(&s_ctr[reason == TERM_LIGHT ? DC_TERM_LIGHT
                                     : reason == TERM_ABSORB ? DC_TERM_ABSORB : DC_TERM_DEPTH], 1u);
                    if (P.path_pixel) path_log_end(P, slot, (int)bounce, reason);
                }
            }
        }
        // compaction: the surviving paths go to [0, n) of the other queue — ballot + prefix popc + ONE atomic per warp.
        // (Finished paths are not replaced here: the launch's last CTA hands out the next iteration's fresh work.)
        const unsigned mc = __ballot_sync(0xffffffffu, cont);
        if (mc) {
            unsigned base = 0u;
            if (lane == 0) base = atomicAdd(&W.st->cnt[cur ^ 1][0], (unsigned)__popc(mc));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (cont) {
                float4* q = qn + 3 * (size_t)(base + __popc(mc & ((1u << lane) - 1u)));
                q[0] = a; q[1] = b; q[2] = c;
            }
        }
    }
    if (n_direct) atomicAdd(&s_ctr[DC_DIRECT], n_direct);
    return 0u;
}

template <bool GEN, bool VIEWS>
__global__ void __launch_bounds__(256, GEN ? 1 : 0) wf_shade(const __grid_constant__ WaveParams W) {
    if (W.st->mode != MODE_RUN) return;        // only this kernel's LAST CTA (below) or the tail ever change the mode
    TraceScope trace(W.trace);
    const RenderParams& P = W.base;
    __shared__ unsigned s_ctr[DC_COUNT];
    if (threadIdx.x < DC_COUNT) s_ctr[threadIdx.x] = 0;
    __syncthreads();
    wf_shade_body<GEN, VIEWS>(W, &W.base.sc, grid_scope(), W.cur, s_ctr);
    __syncthreads();
    if (threadIdx.x < DC_COUNT && s_ctr[threadIdx.x]) atomicAdd(&P.counters[threadIdx.x], (unsigned long long)s_ctr[threadIdx.x]);
    // The last CTA to finish hands out the next iteration's fresh work: the free slots of the other queue, as many as the
    // shared (sample, pixel) counter still has — one returning atomic per LAUNCH (it used to be one per warp and tile).
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&W.st->done, 1u) == gridDim.x - 1) {
            __threadfence();
            W.st->done = 0;
            const unsigned n_cont = *(volatile unsigned*)&W.st->cnt[W.cur ^ 1][0];
            const unsigned want = (unsigned)W.capacity - n_cont;
            unsigned n_fresh = 0;
            unsigned long long base = 0ull;
            if (!W.st->exhausted && want) {
                base = atomicAdd(P.work_counter, (unsigned long long)want);
                if (base < P.total_work) n_fresh = (unsigned)min((unsigned long long)want, P.total_work - base);
                if (base + want >= P.total_work) W.st->exhausted = 1u;
            }
            W.st->cnt[W.cur ^ 1][1] = n_fresh;
            W.st->gen_base[W.cur ^ 1] = base;
            if (n_fresh) atomicAdd(&P.counters[DC_SAMPLES], (unsigned long long)n_fresh);
            if (n_cont + n_fresh == 0) W.st->mode = MODE_DONE;   // kernels already queued behind this one return at once
            __threadfence();
            publish_status(W, n_cont + n_fresh, n_fresh, W.st->exhausted, W.st->mode, W.iter);
        }
    }
}

struct TraceParamsB {
    DevScene sc;
    int n;
    const float* origins;
    const float* dirs;
    const float* times;   // may be null
    double tmin, tmax;
    double* out_t;
    int* out_id;
    unsigned long long* stats;   // may be null: += leaf tests, box tests
};

// ------------------------------------------------------------------------------------------
// RT_ACCEL_BVH: the reference's own accelerator (AABB.hit? hitable.clj:36-48, bvh-node.hit? :97-106, make-bvh :108-123) as
// a flattened tree walked with a short stack.  The boxes are only a CULL, like the FP32 sphere cull of the brute-force
// path: conservative FP32 slab tests (boxes widened at build, NaN-safe min / max, the far bound relaxed by a few ulps),
// and every leaf that survives goes through the same exact FP64 test with the same tie rule — so the closest hit is
// the brute-force one, bit for bit (the reference's tree answers exact ties by tree position and misses a leaf whose
// slab test divides 0 by 0; neither can be observed outside coincident geometry).
// ------------------------------------------------------------------------------------------
struct BvhHit {
    double t;
    int k;
    unsigned tie;
    unsigned n_leaf, n_node;
};
template <bool GEN>
__device__ __forceinline__ BvhHit bvh_closest(const DevScene* sc, float ox, float oy, float oz, float dx, float dy, float dz, float time,
                                              double tmin, double tmax, bool has_ctx, uint2 key, uint32_t pixel, uint32_t sample,
                                              uint32_t bounce) {
    BvhHit H{CUDART_INF, -1, 0xffffffffu, 0u, 0u};
    const float ix = 1.0f / dx, iy = 1.0f / dy, iz = 1.0f / dz;
    // the rounding of (box - origin) is relative to the larger operand: the boxes carry their own share (widened at
    // build), the ray's share widens every box here
    const float e = 2.4e-7f * fmaxf(fmaxf(fabsf(ox), fabsf(oy)), fabsf(oz));
    const float tlo = (float)tmin * (1.0f - 1e-6f);
    float thi = tmax >= (double)FLT_MAX ? FLT_MAX : __double2float_ru(tmax);
    int stack[48];
    int sp = 0, node = 0;
    for (;;) {
        if (node >= 0) {
            const float4 A = __ldg(&sc->bvh[4 * node]), B = __ldg(&sc->bvh[4 * node + 1]), C = __ldg(&sc->bvh[4 * node + 2]);
            const int4 D = __ldg(reinterpret_cast<const int4*>(&sc->bvh[4 * node + 3]));
            H.n_node += 2;
            // slab test of both children; fminf / fmaxf drop a NaN (0 * inf) operand, which keeps the test conservative
            float a0 = ((A.x - e) - ox) * ix, a1 = ((A.w + e) - ox) * ix, b0 = ((A.y - e) - oy) * iy, b1 = ((B.x + e) - oy) * iy,
                  c0 = ((A.z - e) - oz) * iz, c1 = ((B.y + e) - oz) * iz;
            float ln = fmaxf(fmaxf(fminf(a0, a1), fminf(b0, b1)), fmaxf(fminf(c0, c1), tlo));
            float lf = fminf(fminf(fmaxf(a0, a1), fmaxf(b0, b1)), fminf(fmaxf(c0, c1), thi));
            a0 = ((B.z - e) - ox) * ix; a1 = ((C.y + e) - ox) * ix; b0 = ((B.w - e) - oy) * iy; b1 = ((C.z + e) - oy) * iy;
            c0 = ((C.x - e) - oz) * iz; c1 = ((C.w + e) - oz) * iz;
            float rn = fmaxf(fmaxf(fminf(a0, a1), fminf(b0, b1)), fmaxf(fminf(c0, c1), tlo));
            float rf = fminf(fminf(fmaxf(a0, a1), fmaxf(b0, b1)), fminf(fmaxf(c0, c1), thi));
            const bool hl = ln <= lf * 1.0000005f + 1e-30f, hr = rn <= rf * 1.0000005f + 1e-30f;
            if (hl && hr) {                      // nearer child first, the other on the stack
                const bool left_first = ln <= rn;
                stack[sp++] = left_first ? D.y : D.x;
                node = left_first ? D.x : D.y;
                continue;
            }
            if (hl) { node = D.x; continue; }
            if (hr) { node = D.y; continue; }
        } else {
            const int k = ~node;
            H.n_leaf++;
            const double t = refine_leaf<GEN>(sc, k, ox, oy, oz, dx, dy, dz, time, tmin, tmax, has_ctx, key, pixel, sample, bounce);
            if (t < CUDART_INF) {
                const unsigned tie = __ldg(&sc->tie_hi[k]);
                if (t < H.t || (t == H.t && tie < H.tie)) {
                    H.t = t; H.k = k; H.tie = tie;
                    thi = fminf(thi, __double2float_ru(t));   // boxes entirely beyond the hit are skipped; equal t still passes (ties)
                }
            }
        }
        if (sp == 0) break;
        node = stack[--sp];
    }
    return H;
}

// one wavefront iteration's closest-hit search through the BVH: replaces wf_cull + wf_refine + wf_tiebreak.  One thread
// per entry: load (or, for a fresh entry, generate) the ray, walk the tree, leave (t, key) in the closest-hit words for
// wf_shade.  The direct spheres stay with wf_shade as in the brute-force path.
template <bool GEN, bool VIEWS>
__global__ void __launch_bounds__(128, GEN ? 1 : 0) wf_bvh(const __grid_constant__ WaveParams W) {
    if (W.st->mode != MODE_RUN) return;
    TraceScope trace(W.trace);
    const RenderParams& P = W.base;
    __shared__ unsigned s_ctr[DC_COUNT];
    if (threadIdx.x < DC_COUNT) s_ctr[threadIdx.x] = 0;
    __syncthreads();
    const int cur = W.cur;
    const unsigned n_g = W.st->cnt[cur][0], n_p = W.st->cnt[cur][1], n = n_g + n_p, p0 = (unsigned)W.capacity - n_p;
    const unsigned long long gen_base = W.st->gen_base[cur];
    float4* qc = cur ? W.queue[1] : W.queue[0];
    unsigned n_leaf = 0, n_node = 0;
    for (unsigned v = blockIdx.x * blockDim.x + threadIdx.x; v < n; v += gridDim.x * blockDim.x) {
        float4 a, b, c;
        unsigned idx;
        if (v >= n_g) {
            idx = p0 + (v - n_g);
            make_path<VIEWS>(P, gen_base + (v - n_g), a, b, c);
            float4* q = qc + 3 * (size_t)idx;
            q[0] = a; q[1] = b; q[2] = c;
        } else {
            idx = v;
            a = qc[3 * (size_t)idx]; b = qc[3 * (size_t)idx + 1]; c = qc[3 * (size_t)idx + 2];
        }
        const uint32_t sd = __float_as_uint(c.w);
        const BvhHit H = bvh_closest<GEN>(&W.base.sc, a.x, a.y, a.z, b.x, b.y, b.z, a.w, 0.001, (double)FLT_MAX, true, P.key,
                                          rng_pixel<VIEWS>(P, __float_as_uint(b.w)), sd >> 8, (uint32_t)(P.max_depth - (int)(sd & 255u) + 1));
        n_leaf += H.n_leaf; n_node += H.n_node;
        if (H.k >= 0) {
            W.best_t[idx] = (unsigned long long)__double_as_longlong(H.t);
            W.best_key[idx] = ((unsigned long long)H.tie << 32) | (unsigned)H.k;
        }
    }
    atomicAdd(&s_ctr[DC_CANDIDATES], n_leaf);
    atomicAdd(&s_ctr[DC_BVH_NODES], n_node);
    __syncthreads();
    if (threadIdx.x < DC_COUNT && s_ctr[threadIdx.x]) atomicAdd(&P.counters[threadIdx.x], (unsigned long long)s_ctr[threadIdx.x]);
    if (blockIdx.x == 0 && threadIdx.x == 0) {   // the housekeeping wf_cull / wf_refine do in the brute-force path
        atomicAdd(&P.counters[DC_RAYS], (unsigned long long)n);
        W.st->batch = 0;
        W.st->npairs = 0;
        W.st->cnt[cur ^ 1][0] = 0;
        W.st->cnt[cur ^ 1][1] = 0;
    }
}

// rt_trace_primary through the BVH (one thread per ray; the direct spheres are tested exactly, after the tree)
template <bool GEN>
__global__ void __launch_bounds__(128) trace_bvh_kernel(const __grid_constant__ TraceParamsB P) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= P.n) return;
    const float ox = P.origins[3 * idx], oy = P.origins[3 * idx + 1], oz = P.origins[3 * idx + 2];
    const float dx = P.dirs[3 * idx], dy = P.dirs[3 * idx + 1], dz = P.dirs[3 * idx + 2];
    const float tm = P.times ? P.times[idx] : 0.f;
    BvhHit H = bvh_closest<GEN>(&P.sc, ox, oy, oz, dx, dy, dz, tm, P.tmin, P.tmax, false, make_uint2(0u, 0u), 0u, 0u, 0u);
    for (int k = P.sc.n_list; k < P.sc.n; ++k) {
        const double t = refine_leaf<GEN>(&P.sc, k, ox, oy, oz, dx, dy, dz, tm, P.tmin, P.tmax, false, make_uint2(0u, 0u), 0u, 0u, 0u);
        const unsigned tie = __ldg(&P.sc.tie_hi[k]);
        if (t < H.t || (t < CUDART_INF && t == H.t && tie < H.tie)) { H.t = t; H.k = k; H.tie = tie; }
    }
    P.out_t[idx] = H.t;
    P.out_id[idx] = H.k >= 0 ? __ldg(&P.sc.orig_id[H.k]) : -1;
    if (P.stats) {
        atomicAdd(&P.stats[0], (unsigned long long)H.n_leaf);
        atomicAdd(&P.stats[1], (unsigned long long)H.n_node);
    }
}

// The thin end of a tail slice: a few dozen paths with up to max_depth bounces still to go (on the random scene a late
// bounce ends only ~8 % of the paths).  Staged, every bounce of those few paths costs the CTA four barriers and a chain of
// dependent global loads (pairs -> ray -> sphere -> closest-hit words -> candidates -> queue record: ~12 us per bounce
// whatever the population, RT_TAIL_DIAG); here a GROUP of `lpp` lanes (8 | 16 | 32: 4 | 2 | 1 paths per warp) takes one
// path at a time and keeps it in registers until it ends.  All lanes of a group hold the same ray; the listed leaves are
// dealt over the group's lanes (the same conservative FP32 key as the cull, then the exact FP64 test for what passed,
// with the warp converged), the direct spheres likewise, the closest hit is the minimum over the group of (t bits, tie
// key) — the merge rule of wf_refine + wf_tiebreak + wf_shade — and the shading runs on every lane of the group with
// identical inputs (same Philox block); the group's first lane owns the side effects.  A group whose path has ended
// claims the next one from the slice's shared counter.  Same arithmetic as the staged path: results equal bit for bit.
template <bool GEN, bool VIEWS>
__device__ __forceinline__ void wf_solo_paths(const WaveParams& W, const DevScene* scp, const float4* qc, unsigned n, unsigned* claim,
                                              const float4* s_cull, unsigned* s_ctr) {
    const RenderParams& P = W.base;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lpp = W.tail_lpp;                       // lanes per path: 8, 16 or 32
    const unsigned sub = lane & (lpp - 1u), lead = lane & ~(lpp - 1u);
    bool active = false;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a, c = a;
    uint32_t slot = 0u, pix = 0u;
    unsigned n_rays = 0, n_cand = 0, n_direct = 0;
    for (;;) {
        // every collective below is executed by the whole warp; a group without a path just idles through the bounce
        unsigned i = 0xffffffffu;
        if (!active && sub == 0u) i = atomicAdd(claim, 1u);
        i = __shfl_sync(0xffffffffu, i, (int)lead);
        if (!active && i < n) {
            a = qc[3 * (size_t)i]; b = qc[3 * (size_t)i + 1]; c = qc[3 * (size_t)i + 2];
            slot = __float_as_uint(b.w);
            pix = rng_pixel<VIEWS>(P, slot);
            active = true;
        }
        if (!__any_sync(0xffffffffu, active)) break;
        const uint32_t sd = __float_as_uint(c.w), smp = sd >> 8;
        const int depth = (int)(sd & 255u);
        const uint32_t bounce = (uint32_t)(P.max_depth - depth + 1);
        Culler<1, 32, false> K;
        K.set_ray(0, a.x, a.y, a.z, b.x, b.y, b.z);
        if (active && sub == 0u) ++n_rays;
        unsigned long long bt = BEST_T_INIT, bkey = BEST_KEY_MISS;
        // 64 * lpp leaves at a time: the cull key of this lane's 64 of them first (bit j = leaf base + lpp j + sub passed; a
        // direct sphere always does), then the exact tests with the warp converged — as many rounds as the busiest lane has
        // candidates (1 or 2), not one round per leaf position that saw a survivor
        for (int base = 0; base < P.sc.n; base += 64 * (int)lpp) {
            unsigned long long mask = 0ull;
            if (active) {
                const int jn = min(64, (P.sc.n - base + (int)lpp - 1) / (int)lpp);
#pragma unroll 4
                for (int j = 0; j < jn; ++j) {
                    const int s = base + (int)lpp * j + (int)sub;
                    bool pass = s < P.sc.n;                       // beyond the list: a sphere that bypasses the cull
                    if (s < P.sc.n_list) {
                        const float4 S = P.preloaded ? s_cull[s] : __ldg(&P.sc.cull_a[s]);
                        pass = (int)K.key_bits(S, 0) >= 0;        // sign bit clear = survived the cull
                    }
                    mask |= (unsigned long long)(pass ? 1u : 0u) << j;
                }
            }
            while (__any_sync(0xffffffffu, mask != 0ull)) {
                if (mask) {
                    const int s = base + (int)lpp * (__ffsll((long long)mask) - 1) + (int)sub;
                    mask &= mask - 1ull;
                    if (s < P.sc.n_list) ++n_cand; else ++n_direct;
                    const double t = refine_leaf<GEN>(scp, s, a.x, a.y, a.z, b.x, b.y, b.z, a.w, 0.001, (double)FLT_MAX, true, P.key, pix, smp,
                                                      bounce);   // core.clj:25 t-range
                    const unsigned long long tb = (unsigned long long)__double_as_longlong(t);
                    const unsigned long long kk = (((unsigned long long)__ldg(&P.sc.tie_hi[s])) << 32) | (unsigned)s;
                    if (t < CUDART_INF && (tb < bt || (tb == bt && kk < bkey))) { bt = tb; bkey = kk; }
                }
            }
        }
        for (unsigned dlt = lpp >> 1; dlt; dlt >>= 1) {    // t > 0: the order of the bit patterns is the order of the values
            const unsigned long long ot = __shfl_xor_sync(0xffffffffu, bt, (int)dlt), ok = __shfl_xor_sync(0xffffffffu, bkey, (int)dlt);
            if (ot < bt || (ot == bt && ok < bkey)) { bt = ot; bkey = ok; }
        }
        if (active) {
            const bool hit = bkey != BEST_KEY_MISS;
            const int k = (int)(unsigned)bkey;
            const double td = __longlong_as_double((long long)bt);
            if (P.path_pixel && sub == 0u) path_log_ray(P, slot, (int)bounce - 1, a, b, hit ? k : -1, hit ? td : CUDART_INF);
            int reason = TERM_MISS;                         // core.clj:40-41 miss -> accum (black)
            bool cont = false;
            if (hit) {
                float3 o = f3(a.x, a.y, a.z), d = f3(b.x, b.y, b.z);
                float3 att, em;
                float tmv = a.w;
                ScatterRng rng{P.key, pix, smp, bounce, nullptr, nullptr};
                reason = TERM_NONE;
                cont = shade_hit<GEN>(P.sc, scp, k, (float)td, o, d, tmv, depth > 0, rng, att, em, reason);
                if (sub == 0u && (em.x != 0.f || em.y != 0.f || em.z != 0.f)) {   // accum += atten * emitted (core.clj:32-34,37-39)
                    float* dst = P.sum + (size_t)frame_slot<VIEWS>(P, slot) * 3;
                    atomicAdd(dst + 0, c.x * em.x);
                    atomicAdd(dst + 1, c.y * em.y);
                    atomicAdd(dst + 2, c.z * em.z);
                }
                if (cont) {
                    a = make_float4(o.x, o.y, o.z, tmv);
                    b = make_float4(d.x, d.y, d.z, b.w);
                    c = make_float4(c.x * att.x, c.y * att.y, c.z * att.z, __uint_as_float((smp << 8) | (uint32_t)(depth - 1)));
                }
            }
            if (!cont) {
                if (sub == 0u) {
                    atomicAdd(&s_ctr[reason == TERM_MISS ? DC_TERM_MISS : reason == TERM_LIGHT ? DC_TERM_LIGHT
                                     : reason == TERM_ABSORB ? DC_TERM_ABSORB : DC_TERM_DEPTH], 1u);
                    if (P.path_pixel) path_log_end(P, slot, (int)bounce, reason);
                }
                active = false;
            }
        }
    }
    if (n_rays) atomicAdd(&s_ctr[DC_RAYS], n_rays);
    if (n_cand) atomicAdd(&s_ctr[DC_CANDIDATES], n_cand);
    if (n_direct) atomicAdd(&s_ctr[DC_DIRECT], n_direct);
}

// Tail of a render: the work counter is exhausted and the queue is short (up to 50 more bounces of a shrinking
// handful of paths).  ONE launch finishes the lane: the queue is cut into one slice per CTA, and every CTA runs
// the wavefront stages on its own slice by itself — its queue counters live in shared memory, the stages are
// separated by __syncthreads() (tens of cycles) instead of kernel boundaries (~8 us of launch floors per
// iteration) or grid.sync() (the cooperative form of this kernel: ~20 us per iteration, 0.75 ms per render).
// The slices are the CTA's ranges of the lane's own buffers, so a slice's population can only shrink in place.
constexpr int kPairsPerEntry = 8;       // pair buffer = 8 (ray, sphere) pairs per queue entry (measured mean: 1.5)
// TR: rays per thread of the tail's cull while a slice is still long (the first bounces after the hand-over, when a
// slice holds thousands of paths): TR = 4 runs them like wf_cull does (4 independent chains per thread), the short-queue
// forms (1 ray per thread, sphere list split across warps) take over as the slice shrinks.
template <int BLOCK, bool GEN, int TR, bool VIEWS>
__global__ void __launch_bounds__(BLOCK, GEN ? 1 : 2) wf_tail(const __grid_constant__ WaveParams W) {
    const RenderParams& P = W.base;
    extern __shared__ float4 smem_f4[];
    float4* s_cull = smem_f4;
    uint32_t* s_list = reinterpret_cast<uint32_t*>(smem_f4 + P.cull_cap);
    __shared__ unsigned s_ctr[DC_COUNT];
    __shared__ WaveState s_st;
    if (W.st->mode == MODE_DONE) return;             // the iterations queued ahead of this launch already drained the lane
    TraceScope trace(W.trace);
    int cur = W.cur;
    const unsigned n_all = W.st->cnt[cur][0];        // the host launches it only once the fresh region stays empty
    const unsigned K = ((n_all + gridDim.x - 1) / gridDim.x + 31u) / 32u * 32u;      // slice capacity
    const unsigned first = blockIdx.x * K;
    if (first < n_all) {                                                              // CTA-uniform
        if (threadIdx.x < DC_COUNT) s_ctr[threadIdx.x] = 0;
        if (threadIdx.x == 0) {
            s_st.cnt[cur][0] = min(K, n_all - first);
            s_st.cnt[cur ^ 1][0] = 0;
            s_st.cnt[0][1] = s_st.cnt[1][1] = 0;
            s_st.gen_base[0] = s_st.gen_base[1] = 0ull;
            s_st.batch = 0;
            s_st.npairs = 0;
            s_st.exhausted = 1;
            s_st.done = 0;
            s_st.mode = MODE_RUN;
            s_st.pad = 0;
        }
        // this CTA's view of the lane's buffers
        const unsigned warps = BLOCK / 32;
        WaveParams L = W;
        L.queue[0] = W.queue[0] + 3 * (size_t)first;
        L.queue[1] = W.queue[1] + 3 * (size_t)first;
        L.best_t = W.best_t + first;
        L.best_key = W.best_key + first;
        L.pairs = W.pairs + (size_t)first * kPairsPerEntry;
        // the slice's share of the pair buffer ends where the allocation ends (the last slice may be cut short)
        L.pair_cap = min(K, (unsigned)W.capacity - first) * kPairsPerEntry;
        const size_t cand_slice = (size_t)wf_cand_region(L, warps) * warps;
        L.cands = W.cands + (size_t)blockIdx.x * cand_slice;
        L.cand_t = W.cand_t + (size_t)blockIdx.x * cand_slice;
        L.cand_count = W.cand_count + blockIdx.x * warps;
        L.st = &s_st;
        L.status = nullptr;
        L.capacity = (int)K;
        L.claims_per_warp = 0;
        L.resident_warps = 0;
        if (P.preloaded) preload_scene(P.sc, s_cull, BLOCK);
        const Scope solo{0u, 1u};
        for (;;) {
            __syncthreads();
            const unsigned n = *(volatile unsigned*)&s_st.cnt[cur][0];
#ifdef RT_TAIL_DIAG
            const bool diag = (blockIdx.x == 0 || blockIdx.x == gridDim.x / 2) && threadIdx.x == 0;
            unsigned long long dt0 = global_timer_ns();
#endif
            if (n <= W.tail_solo) {   // the thin end (or nothing): one warp per path, no more barriers (s_st.done: the claim counter)
                if (n) wf_solo_paths<GEN, VIEWS>(L, &W.base.sc, cur ? L.queue[1] : L.queue[0], n, &s_st.done, s_cull, s_ctr);
#ifdef RT_TAIL_DIAG
                __syncthreads();
                if (diag) printf("tail cta %u solo n %u: %llu ns\n", blockIdx.x, n, global_timer_ns() - dt0);
#endif
                break;
            }
            wf_cull_body<TR, BLOCK, VIEWS>(L, solo, cur, n, 0u, 0ull, s_cull, nullptr, s_list);
            __syncthreads();
#ifdef RT_TAIL_DIAG
            unsigned long long dt1 = global_timer_ns();
            const unsigned np_ = s_st.npairs;
#endif
            wf_refine_body<GEN, VIEWS>(L, &W.base.sc, solo, cur);
            __syncthreads();
#ifdef RT_TAIL_DIAG
            unsigned long long dt2 = global_timer_ns();
#endif
            wf_tiebreak_body(L, solo);
            __syncthreads();
#ifdef RT_TAIL_DIAG
            unsigned long long dt3 = global_timer_ns();
#endif
            wf_shade_body<GEN, VIEWS>(L, &W.base.sc, solo, cur, s_ctr);
#ifdef RT_TAIL_DIAG
            __syncthreads();
            if (diag) printf("tail cta %u n %u pairs %u: cull %llu refine %llu tie %llu shade %llu ns\n", blockIdx.x, n, np_, dt1 - dt0, dt2 - dt1, dt3 - dt2, global_timer_ns() - dt3);
#endif
            cur ^= 1;
        }
        __syncthreads();
        if (threadIdx.x < DC_COUNT && s_ctr[threadIdx.x]) atomicAdd(&P.counters[threadIdx.x], (unsigned long long)s_ctr[threadIdx.x]);
    }
    // the last CTA to finish marks the lane drained: every kernel queued behind this one returns at once
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&W.st->done, 1u) == gridDim.x - 1) {
            W.st->done = 0;
            W.st->cnt[0][0] = W.st->cnt[0][1] = W.st->cnt[1][0] = W.st->cnt[1][1] = 0;
            W.st->mode = MODE_DONE;
            __threadfence();
            publish_status(W, 0u, 0u, 1u, MODE_DONE, W.iter);
        }
    }
}


// ------------------------------------------------------------------------------------------
// Persistent megakernel with path regeneration (kept for comparison): every thread owns R path
// slots; a slot whose path ended pulls the next (sample, pixel) work item (warp-aggregated atomic:
// ballot + prefix popc) so the intersect loop runs with full lanes until the work runs out.
// Warps run asynchronously through generate / intersect / refine / shade code.
// ------------------------------------------------------------------------------------------
// One shared body for the shading of every path slot of the megakernel.  Inlined once per slot (RT_FOR_R) the R copies
// were contracted / scheduled differently, so a path's last bits depended on WHICH slot the dynamic work counter gave
// it — the run-to-run "one path in ~600 k takes a different number of bounces" of the register-capped build of round 1
// (no race: every per-path value lives in registers, everything shared is read-only or atomic).  A single out-of-line
// copy makes the result a function of (pixel, sample) alone.  By value in, one struct out (no caller registers forced
// into local memory).
struct MegaShade {
    float4 o_t;      // scattered origin, ray time
    float4 d_c;      // scattered direction, continue flag (1 / 0)
    float4 att_r;    // attenuation, termination reason
    float4 em;       // emitted
};
template <bool GEN>
__device__ __noinline__ MegaShade mega_shade_one(const DevScene* scp, int k, float t, float ox, float oy, float oz, float dx, float dy,
                                                 float dz, float time, int allow_scatter, uint2 key, uint32_t pix, uint32_t smp,
                                                 uint32_t bounce) {
    float3 o = f3(ox, oy, oz), d = f3(dx, dy, dz), att, em;
    int reason = TERM_NONE;
    ScatterRng rng{key, pix, smp, bounce, nullptr, nullptr};
    const bool cont = shade_hit<GEN>(*scp, scp, k, t, o, d, time, allow_scatter != 0, rng, att, em, reason);
    MegaShade m;
    m.o_t = make_float4(o.x, o.y, o.z, time);
    m.d_c = make_float4(d.x, d.y, d.z, cont ? 1.f : 0.f);
    m.att_r = make_float4(att.x, att.y, att.z, (float)reason);
    m.em = make_float4(em.x, em.y, em.z, 0.f);
    return m;
}

template <int R, int BLOCK, bool GEN, bool VIEWS>
__device__ __forceinline__ void mega_body(const RenderParams& P) {
    extern __shared__ float4 smem_f4[];
    float4* s_cull = smem_f4;
    uint32_t* s_list = reinterpret_cast<uint32_t*>(smem_f4 + P.cull_cap);
    __shared__ unsigned s_ctr[DC_COUNT];
    if (threadIdx.x < DC_COUNT) s_ctr[threadIdx.x] = 0;
    if (P.preloaded) preload_scene(P.sc, s_cull, BLOCK);
    __syncthreads();

    Culler<R, BLOCK> K;
    RefineSink<R, BLOCK, GEN> I;
    I.tmin = 0.001;               // core.clj:25
    I.tmax = (double)FLT_MAX;     // Float/MAX_VALUE
    I.ncand = 0;
    I.sc = &P.sc;
    I.has_ctx = true;
    I.key = P.key;

    float ar[R], ag[R], ab[R];    // attenuation (core.clj:23 `atten`); the rays themselves live in the sink
    uint32_t slot[R];             // where the path's radiance goes: the pixel (a render) / the path (rt_trace_paths)
    uint32_t (&pix)[R] = I.pix, (&smp)[R] = I.smp;
    int depth[R];
    bool alive[R];
    RT_FOR_R { alive[r] = false; I.ox[r] = I.oy[r] = I.oz[r] = I.tm[r] = 0.f; I.dx[r] = 1.f; I.dy[r] = I.dz[r] = 0.f; pix[r] = smp[r] = slot[r] = 0u; I.bounce[r] = 0u; }
    unsigned n_rays = 0, n_samples = 0, n_direct = 0;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned pshard = (unsigned)P.nx * (unsigned)P.rows_in_shard;

    for (;;) {
        // ---- generate: refill dead slots -----------------------------------------------------
        RT_FOR_R {
            unsigned need = __ballot_sync(0xffffffffu, !alive[r]);
            if (need) {
                int leader = __ffs(need) - 1;
                unsigned long long base = 0;
                if ((int)lane == leader) base = atomicAdd(P.work_counter, (unsigned long long)__popc(need));
                base = __shfl_sync(0xffffffffu, base, leader);
                unsigned long long w = base + __popc(need & ((1u << lane) - 1u));
                if (!alive[r] && w < P.total_work) {
                    unsigned s_local = (unsigned)(w / pshard);
                    unsigned q = (unsigned)(w - (unsigned long long)s_local * pshard);
                    int row_local = (int)(q / (unsigned)P.nx);
                    int i = (int)(q - (unsigned)row_local * (unsigned)P.nx);
                    int j = P.row_offset + row_local * P.row_stride;
                    pix[r] = (uint32_t)j * (uint32_t)P.nx + (uint32_t)i;
                    smp[r] = (uint32_t)(P.sample_begin + (int)s_local);
                    slot[r] = pix[r];
                    if (P.path_pixel) {                       // rt_trace_paths: work item w is path w of the caller's list
                        pix[r] = (uint32_t)__ldg(&P.path_pixel[w]);
                        smp[r] = (uint32_t)__ldg(&P.path_sample[w]);
                        j = (int)(pix[r] / (uint32_t)P.nx);
                        i = (int)(pix[r] - (uint32_t)j * (uint32_t)P.nx);
                        slot[r] = (uint32_t)w;
                    }
                    float3 o, d;
                    if (VIEWS && P.views && !P.path_pixel) {   // rt_render_views: as make_path
                        const uint32_t v = view_of(P, slot[r]);
                        pix[r] = slot[r] - v * P.view_px;
                        const CameraRay cr = view_ray(P.views, v, P.nx, P.ny, i, j - (int)v * P.ny, pix[r], smp[r], P.key);
                        o = cr.o; d = cr.d; I.tm[r] = cr.time;
                    } else {
                        generate_ray(P.cam, P.nx, P.ny, i, j, pix[r], smp[r], P.key, o, d, I.tm[r], nullptr);
                    }
                    I.ox[r] = o.x; I.oy[r] = o.y; I.oz[r] = o.z;
                    I.dx[r] = d.x; I.dy[r] = d.y; I.dz[r] = d.z;
                    ar[r] = ag[r] = ab[r] = 1.0f;
                    depth[r] = P.max_depth;
                    alive[r] = true;
                    n_samples++;
                }
            }
        }
        bool any_alive = false;
        RT_FOR_R any_alive |= alive[r];
        // preloaded scene: warps are independent (no CTA barrier inside the loop) and leave on their own;
        // tiled scene: the tile loads need every thread of the CTA
        if (P.preloaded) {
            if (!__any_sync(0xffffffffu, any_alive)) break;
        } else {
            if (!__syncthreads_or(any_alive)) break;
        }

        // ---- intersect ----------------------------------------------------------------------------
        unsigned live = 0;
        RT_FOR_R {
            if (alive[r]) { K.set_ray(r, I.ox[r], I.oy[r], I.oz[r], I.dx[r], I.dy[r], I.dz[r]); n_rays++; live |= 1u << r; }
            else K.kill(r);
            I.bounce[r] = (uint32_t)(P.max_depth - depth[r] + 1);
        }
        I.begin();
        K.run(P.sc, s_cull, P.cull_cap, P.preloaded != 0, s_list, I);
        n_direct += I.direct(live);

        // ---- shade ------------------------------------------------------------------------------
        RT_FOR_R {
            if (alive[r]) {
                if (P.path_pixel)
                    path_log_ray(P, slot[r], (int)I.bounce[r] - 1, make_float4(I.ox[r], I.oy[r], I.oz[r], I.tm[r]),
                                 make_float4(I.dx[r], I.dy[r], I.dz[r], 0.f), I.best_k[r], I.best_t[r]);
                if (I.best_k[r] < 0) {                       // core.clj:40-41 miss -> accum (black)
                    alive[r] = false;
                    atomicAdd(&s_ctr[DC_TERM_MISS], 1u);
                    if (P.path_pixel) path_log_end(P, slot[r], (int)I.bounce[r], TERM_MISS);
                } else {
                    const MegaShade ms = mega_shade_one<GEN>(&P.sc, I.best_k[r], (float)I.best_t[r], I.ox[r], I.oy[r], I.oz[r], I.dx[r], I.dy[r],
                                                             I.dz[r], I.tm[r], depth[r] > 0 ? 1 : 0, P.key, pix[r], smp[r], I.bounce[r]);
                    const float3 o = f3(ms.o_t.x, ms.o_t.y, ms.o_t.z), d = f3(ms.d_c.x, ms.d_c.y, ms.d_c.z);
                    const float3 att = f3(ms.att_r.x, ms.att_r.y, ms.att_r.z), em = f3(ms.em.x, ms.em.y, ms.em.z);
                    const bool cont = ms.d_c.w != 0.f;
                    const int reason = (int)ms.att_r.w;
                    I.tm[r] = ms.o_t.w;
                    if (em.x != 0.f || em.y != 0.f || em.z != 0.f) {   // accum += atten * emitted (core.clj:32-34,37-39)
                        float* dst = P.sum + (size_t)slot[r] * 3;
                        atomicAdd(dst + 0, ar[r] * em.x);
                        atomicAdd(dst + 1, ag[r] * em.y);
                        atomicAdd(dst + 2, ab[r] * em.z);
                    }
                    if (cont) {
                        ar[r] *= att.x; ag[r] *= att.y; ab[r] *= att.z;     // core.clj:31
                        I.ox[r] = o.x; I.oy[r] = o.y; I.oz[r] = o.z;
                        I.dx[r] = d.x; I.dy[r] = d.y; I.dz[r] = d.z;
                        depth[r]--;
                    } else {
                        alive[r] = false;
                        atomicAdd(&s_ctr[reason == TERM_LIGHT ? DC_TERM_LIGHT
                                         : reason == TERM_ABSORB ? DC_TERM_ABSORB : DC_TERM_DEPTH], 1u);
                        if (P.path_pixel) path_log_end(P, slot[r], (int)I.bounce[r], reason);
                    }
                }
            }
        }
    }

    atomicAdd(&s_ctr[DC_RAYS], n_rays);
    atomicAdd(&s_ctr[DC_SAMPLES], n_samples);
    atomicAdd(&s_ctr[DC_CANDIDATES], I.ncand);
    atomicAdd(&s_ctr[DC_DIRECT], n_direct);
    __syncthreads();
    if (threadIdx.x < DC_COUNT && s_ctr[threadIdx.x]) atomicAdd(&P.counters[threadIdx.x], (unsigned long long)s_ctr[threadIdx.x]);
}
template <int R, int BLOCK, int MINB, bool GEN>
__global__ void __launch_bounds__(BLOCK, MINB) mega_kernel(const __grid_constant__ RenderParams P) {
    mega_body<R, BLOCK, GEN, false>(P);
}
// the megakernel of a batch of views (rt_render_views); the single-camera one above holds none of the batch code
template <int R, int BLOCK, int MINB, bool GEN>
__global__ void __launch_bounds__(BLOCK, MINB) mega_views_kernel(const __grid_constant__ RenderParams P) {
    mega_body<R, BLOCK, GEN, true>(P);
}

// ------------------------------------------------------------------------------------------
// rt_trace_primary: closest hit of n caller-given rays (same Culler + FP64 refine as the renderer)
// ------------------------------------------------------------------------------------------
struct TraceParams {
    DevScene sc;
    int n;
    const float* origins;
    const float* dirs;
    const float* times;   // may be null
    double tmin, tmax;
    double* out_t;
    int* out_id;
    int cull_cap, preloaded;
};

template <int R, int BLOCK, bool GEN>
__global__ void __launch_bounds__(BLOCK) trace_kernel(const __grid_constant__ TraceParams P) {
    extern __shared__ float4 smem_f4[];
    float4* s_cull = smem_f4;
    uint32_t* s_list = reinterpret_cast<uint32_t*>(smem_f4 + P.cull_cap);
    if (P.preloaded) preload_scene(P.sc, s_cull, BLOCK);
    __syncthreads();
    Culler<R, BLOCK> K;
    RefineSink<R, BLOCK, GEN> I;
    I.tmin = P.tmin;
    I.tmax = P.tmax;
    I.ncand = 0;
    I.sc = &P.sc;
    I.has_ctx = false;            // no path behind these rays: a ConstantMedium draws 0.5
    for (long long base = (long long)blockIdx.x * BLOCK * R; base < P.n; base += (long long)gridDim.x * BLOCK * R) {
        unsigned live = 0;
        RT_FOR_R {
            long long idx = base + (long long)r * BLOCK + threadIdx.x;
            if (idx < P.n) {
                I.ox[r] = P.origins[3 * idx]; I.oy[r] = P.origins[3 * idx + 1]; I.oz[r] = P.origins[3 * idx + 2];
                I.dx[r] = P.dirs[3 * idx]; I.dy[r] = P.dirs[3 * idx + 1]; I.dz[r] = P.dirs[3 * idx + 2];
                I.tm[r] = P.times ? P.times[idx] : 0.f;
                K.set_ray(r, I.ox[r], I.oy[r], I.oz[r], I.dx[r], I.dy[r], I.dz[r]);
                live |= 1u << r;
            } else {
                I.ox[r] = I.oy[r] = I.oz[r] = I.tm[r] = 0.f;
                I.dx[r] = 1.f; I.dy[r] = 0.f; I.dz[r] = 0.f;
                K.kill(r);
            }
        }
        I.begin();
        K.run(P.sc, s_cull, P.cull_cap, P.preloaded != 0, s_list, I);
        I.direct(live);
        RT_FOR_R {
            long long idx = base + (long long)r * BLOCK + threadIdx.x;
            if (idx < P.n) {
                P.out_t[idx] = I.best_t[r];
                P.out_id[idx] = (I.best_k[r] >= 0) ? __ldg(&P.sc.orig_id[I.best_k[r]]) : -1;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// diagnostics
// ------------------------------------------------------------------------------------------
// The cull's contract, checked pair by pair: every (ray, listed sphere) whose exact FP64 test accepts a root in
// (tmin, tmax) must have a clear sign bit in the FP32 key computed by the very code of the hot loop.
// out[0] = pairs the cull would have lost (must be 0), out[1] = cull survivors, out[2] = exact candidates.
__global__ void __launch_bounds__(128) cull_check_kernel(const __grid_constant__ DevScene sc, int n, const float* origins, const float* dirs,
                                                         const float* times, double tmin, double tmax,
                                                         unsigned long long* out) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long lost = 0, surv = 0, cand = 0;
    if (idx < n) {
        const float ox = origins[3 * idx], oy = origins[3 * idx + 1], oz = origins[3 * idx + 2];
        const float dx = dirs[3 * idx], dy = dirs[3 * idx + 1], dz = dirs[3 * idx + 2];
        const float tm = times ? times[idx] : 0.f;
        Culler<1, 128> K;
        K.set_ray(0, ox, oy, oz, dx, dy, dz);
        K.pin();
        for (int k = 0; k < sc.n_list; ++k) {
            const bool culled = (K.key_bits(__ldg(&sc.cull_a[k]), 0) >> 31) != 0u;
            const double t = sc.generic ? refine_leaf<true>(&sc, k, ox, oy, oz, dx, dy, dz, tm, tmin, tmax, false, make_uint2(0u, 0u), 0u, 0u, 0u)
                                        : refine_leaf<false>(&sc, k, ox, oy, oz, dx, dy, dz, tm, tmin, tmax, false, make_uint2(0u, 0u), 0u, 0u, 0u);
            surv += culled ? 0u : 1u;
            if (t < CUDART_INF) {
                cand++;
                lost += culled ? 1u : 0u;
            }
        }
    }
    if (lost) atomicAdd(&out[0], lost);
    if (surv) atomicAdd(&out[1], surv);
    if (cand) atomicAdd(&out[2], cand);
}

// rt_sample_device: the closed-form samplers by themselves (util.clj:32-52), keyed (pixel = index, sample 0)
__global__ void sampler_kernel(int kind, int n, uint2 key, float* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (kind == 0) {
        const float3 p = rand_in_unit_sphere(key, (uint32_t)i, 0u, 1u, 1u);
        out[3 * i] = p.x; out[3 * i + 1] = p.y; out[3 * i + 2] = p.z;
    } else {
        const float2 p = rand_in_unit_disk(key, (uint32_t)i, 0u, 1u);
        out[2 * i] = p.x; out[2 * i + 1] = p.y;
    }
}

__global__ void genrays_kernel(DevCamera cam, int n, int nx, int ny, const int* ij, const int* s, uint2 key, float* out_o,
                               float* out_d, float* out_t, float* out_rnd) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    int i = ij[2 * idx], j = ij[2 * idx + 1];
    float3 o, d;
    float tm;
    float rnd[5];
    generate_ray(cam, nx, ny, i, j, (uint32_t)j * (uint32_t)nx + (uint32_t)i, (uint32_t)s[idx], key, o, d, tm, rnd);
    out_o[3 * idx] = o.x; out_o[3 * idx + 1] = o.y; out_o[3 * idx + 2] = o.z;
    out_d[3 * idx] = d.x; out_d[3 * idx + 1] = d.y; out_d[3 * idx + 2] = d.z;
    out_t[idx] = tm;
    if (out_rnd)
        for (int k = 0; k < 5; ++k) out_rnd[5 * idx + k] = rnd[k];
}

__global__ void shade_kernel(const __grid_constant__ DevScene sc, int n, const float* origins, const float* dirs, const float* times,
                             const int* hit_id, const double* hit_t, const float* ball, const float* u01v, float* out_o,
                             float* out_d, float* out_att, float* out_em, int* out_flags) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    float3 o = f3(origins[3 * idx], origins[3 * idx + 1], origins[3 * idx + 2]);
    float3 d = f3(dirs[3 * idx], dirs[3 * idx + 1], dirs[3 * idx + 2]);
    float3 att = f3(0.f, 0.f, 0.f), em = f3(0.f, 0.f, 0.f);
    int flag = -1;
    int id = hit_id[idx];
    if (id >= 0 && id < sc.n) {
        int k = sc.cull_of_orig[id];
        int reason = TERM_NONE;
        ScatterRng rng{make_uint2(0u, 0u), 0u, 0u, 0u, ball + 3 * idx, u01v + idx};
        float tmv = times ? times[idx] : 0.f;
        bool cont = sc.generic ? shade_hit<true>(sc, &sc, k, (float)hit_t[idx], o, d, tmv, true, rng, att, em, reason)
                               : shade_hit<false>(sc, &sc, k, (float)hit_t[idx], o, d, tmv, true, rng, att, em, reason);
        flag = cont ? 1 : 0;
        if (!cont) {
            o = f3(0.f, 0.f, 0.f); d = o; att = o;
        }
    } else {
        o = f3(0.f, 0.f, 0.f); d = o;
    }
    out_o[3 * idx] = o.x; out_o[3 * idx + 1] = o.y; out_o[3 * idx + 2] = o.z;
    out_d[3 * idx] = d.x; out_d[3 * idx + 1] = d.y; out_d[3 * idx + 2] = d.z;
    out_att[3 * idx] = att.x; out_att[3 * idx + 1] = att.y; out_att[3 * idx + 2] = att.z;
    out_em[3 * idx] = em.x; out_em[3 * idx + 1] = em.y; out_em[3 * idx + 2] = em.z;
    out_flags[idx] = flag;
}

// core.clj:52-57: (sum * (1/nr)) -> sqrt -> * 255.99 -> (int (min 255.99 x)); row ny-1-j (core.clj:105).
// Evaluated in double from the float sums so it matches the oracle's resolve bit for bit.
// `peers` (optional): other devices' sum buffers mapped over NVLink peer access, added first.
struct ResolveParams {
    const float* sum;
    const float* peers[7];
    int n_peers;
    int nx, ny, nr;
    int n_views;         // > 1: n_views stacked images of ny rows (rt_render_views), each flipped on its own
    uint8_t* rgb8;       // may be null
    float* mean;         // may be null: (float)(sum / nr), same layout as sum
    float* sum_out;      // may be null: reduced sum written back (multi-device)
};
__global__ void resolve_kernel(const ResolveParams P) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;   // over nx*ny*n_views*3
    int total = P.nx * P.ny * 3 * (P.n_views > 1 ? P.n_views : 1);
    if (idx >= total) return;
    float s = P.sum[idx];
    for (int p = 0; p < P.n_peers; ++p) s += P.peers[p][idx];
    if (P.sum_out) P.sum_out[idx] = s;
    double x = (double)s * (1.0 / (double)P.nr);
    if (P.mean) P.mean[idx] = (float)x;
    if (P.rgb8) {
        int ch = idx % 3, pixel = idx / 3;
        int i = pixel % P.nx, j = pixel / P.nx;
        int row = P.ny - 1 - j;
        if (P.n_views > 1) {   // row j of view v = j / ny lands on row ny - 1 - (j - v ny) of the view's image
            const int v = j / P.ny;
            row += 2 * v * P.ny;
        }
        double y = sqrt(x) * 255.99;
        int v = (y != y) ? 0 : (int)fmin(255.99, y);   // (int NaN) = 0 on the JVM
        P.rgb8[((size_t)row * P.nx + i) * 3 + ch] = (uint8_t)v;
    }
}

// FP32 peak: independent FFMA chains (and the packed FFMA2 form), no memory traffic.
template <bool PACKED>
__global__ void __launch_bounds__(256) ffma_peak_kernel(float* out, int iters, float a, float b) {
    if (PACKED) {
        float2 x[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = make_float2(threadIdx.x * 1e-3f + i, threadIdx.x * 2e-3f - i);
        float2 aa = make_float2(a, a), bb = make_float2(b, b);
        for (int it = 0; it < iters; ++it) {
#pragma unroll
            for (int i = 0; i < 8; ++i) x[i] = __ffma2_rn(x[i], aa, bb);
        }
        float acc = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) acc += x[i].x + x[i].y;
        out[blockIdx.x * blockDim.x + threadIdx.x] = acc;
    } else {
        float x[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) x[i] = threadIdx.x * 1e-3f + i;
        for (int it = 0; it < iters; ++it) {
#pragma unroll
            for (int i = 0; i < 16; ++i) x[i] = fmaf(x[i], a, b);
        }
        float acc = 0.f;
#pragma unroll
        for (int i = 0; i < 16; ++i) acc += x[i];
        out[blockIdx.x * blockDim.x + threadIdx.x] = acc;
    }
}

}  // namespace rt
