// rt_scene_build.cuh — the scene blob of a sphere scene built on the device from per-primitive arrays that already live in
// device memory (rt_set_scene_device).  Every kernel restates one step of rt_set_scene_ex for the sphere-only case
// (no rt_scene_ext: generic = 0, tie rule RT_TIE_HITLIST, no Isotropic material) and writes the bytes the host path
// writes: FP64 with explicitly rounded intrinsics (no FMA contraction), the same float rounding, the same orders.
//
//   sb_validate        one thread per primitive: the host loop's checks (unknown flag bit, material id out of range,
//                      a mover with t1 == t0) as min(4 i + check), the movers' time window, |r| for the median
//   (cub radix sort)   the radii; the median |r| is sorted[n / 2] (nth_element is value-based: the same value).  A
//                      non-negative double orders as its bits do, so both sorts here are the u64-key sort of the BVH build
//   sb_small_partials  per block, in a fixed order: sums of the small spheres' centres and their count
//   sb_candidates      direct-sphere candidates (|r| >= 8 median, |c - centroid| <= 1.05 |r|), in any order
//   sb_direct_choose   one thread: the first 8 candidates by (-|r|, index), then ordered by (-dist / |r|, index)
//   sb_perm            cull order: the listed spheres in caller order, the direct spheres after them
//   sb_gather          one thread per cull entry: geometry, flags, material, orig / cull_of, shading record, tie key and the
//                      FP64 bounding sphere, in the blob's layout
//   (cub radix sort)   listed leaves by bounding radius, descending (key ~bits), stable (the host's std::stable_sort)
//   sb_deal            the tensor-core feature rows: leaf of each row (tc_row_k), padding rows' slots
//   sb_cull_records    one thread per leaf: build_cull_records' FP32 record (and the padding records' W = -inf)
//   sb_tc_rows         one thread per feature row: the leaf's 32 TF32 slots (tc::sphere_slots) in the canonical layout
//
// The centroid of the small spheres is a parallel FP64 sum where the host adds in caller order, so the two can differ in
// the last bit.  That can change which spheres are direct only for a sphere within ~1e-15 (relative) of the 1.05 boundary,
// and the choice changes the work split only, never a result (DESIGN §3).
#pragma once

#include "rt_bvh_build.cuh"
#include "rt_kernels.cuh"   // tc:: (rt_cull_tc.cuh): sphere_slots, padding_slots, canon_off

namespace rt {

constexpr int kSbBlock = 256;
constexpr int kSbPartials = 256;   // blocks of sb_small_partials (fixed: the sum's order depends on n only)
constexpr int kSbMaxDirect = 8;

// what the host reads back before it lays the blob out
struct SbResult {
    unsigned long long err;   // min(4 i + check) over the failing primitives: check 0 flag, 1 material id, 2 t1 == t0; ~0 = none
    unsigned win_lo, win_hi;  // bvh_ordered(min / max of the movers' t0, t1); identities when there is no mover
    int n_direct;
    int direct[kSbMaxDirect]; // caller indices of the direct spheres, in cull order
    double centroid[3];
};

// the per-primitive arrays of rt_scene_desc, as device pointers (center1 / t0t1 / flags may be null)
struct SbInput {
    const float* c0r;
    const float* c1;
    const float* t0t1;
    const unsigned* flags;
    const int* mat;
    int n, n_materials;
};

__device__ __forceinline__ bool sb_moving(const SbInput& in, int i) {
    return in.flags && (in.flags[i] & RT_SPHERE_MOVING) && in.c1 && in.t0t1;
}

__device__ __forceinline__ float sb_round_up_f32(double x) {
    float f = __double2float_rn(x);
    if ((double)f < x) f = nextafterf(f, INFINITY);
    return f;
}

__global__ void __launch_bounds__(kSbBlock) sb_validate(const SbInput in, SbResult* res, double* radii) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= in.n) return;
    const unsigned fl = in.flags ? in.flags[i] : 0u;
    int check = -1;
    if (fl & ~(RT_SPHERE_UV | RT_SPHERE_MOVING)) check = 0;
    else if (in.mat[i] < 0 || in.mat[i] >= in.n_materials) check = 1;
    else if (sb_moving(in, i)) {
        const float t0 = in.t0t1[2 * (size_t)i], t1 = in.t0t1[2 * (size_t)i + 1];
        if (!(t1 != t0)) check = 2;
        atomicMin(&res->win_lo, bvh_ordered(fminf(t0, t1)));
        atomicMax(&res->win_hi, bvh_ordered(fmaxf(t0, t1)));
    }
    if (check >= 0) atomicMin(&res->err, 4ull * (unsigned long long)i + (unsigned long long)check);
    if (radii) radii[i] = fabs((double)in.c0r[4 * (size_t)i + 3]);
}

// partials[4 b + (0, 1, 2, 3)] = sums of x, y, z and the count of the spheres with |r| < 8 median in block b's share
__global__ void __launch_bounds__(kSbBlock) sb_small_partials(const SbInput in, const double* radii, const double* sorted, double* partials) {
    __shared__ double s[4][kSbBlock];
    const double big = __dmul_rn(8.0, sorted[in.n / 2]);
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < in.n; i += gridDim.x * blockDim.x)
        if (radii[i] < big) {
            for (int c = 0; c < 3; ++c) acc[c] = __dadd_rn(acc[c], (double)in.c0r[4 * (size_t)i + c]);
            acc[3] = __dadd_rn(acc[3], 1.0);
        }
    for (int c = 0; c < 4; ++c) s[c][threadIdx.x] = acc[c];
    __syncthreads();
    for (int h = kSbBlock / 2; h > 0; h /= 2) {
        if ((int)threadIdx.x < h)
            for (int c = 0; c < 4; ++c) s[c][threadIdx.x] = __dadd_rn(s[c][threadIdx.x], s[c][threadIdx.x + h]);
        __syncthreads();
    }
    if (threadIdx.x < 4) partials[4 * blockIdx.x + threadIdx.x] = s[threadIdx.x][0];
}

// one block of kSbPartials threads: the centroid cen[c] = sum / max(1, count)
__global__ void __launch_bounds__(kSbPartials) sb_centroid(const double* partials, SbResult* res) {
    __shared__ double s[4][kSbPartials];
    for (int c = 0; c < 4; ++c) s[c][threadIdx.x] = partials[4 * threadIdx.x + c];
    __syncthreads();
    for (int h = kSbPartials / 2; h > 0; h /= 2) {
        if ((int)threadIdx.x < h)
            for (int c = 0; c < 4; ++c) s[c][threadIdx.x] = __dadd_rn(s[c][threadIdx.x], s[c][threadIdx.x + h]);
        __syncthreads();
    }
    if (threadIdx.x < 3) res->centroid[threadIdx.x] = __ddiv_rn(s[threadIdx.x][0], fmax(1.0, s[3][0]));
}

__device__ __forceinline__ double sb_dist(const SbInput& in, int i, const double cen[3]) {
    double d2 = 0.0;
    for (int c = 0; c < 3; ++c) {
        const double x = __dsub_rn((double)in.c0r[4 * (size_t)i + c], cen[c]);
        d2 = __dadd_rn(d2, __dmul_rn(x, x));
    }
    return __dsqrt_rn(d2);
}

__global__ void __launch_bounds__(kSbBlock) sb_candidates(const SbInput in, const double* radii, const double* sorted, const SbResult* res,
                                                          int* cand, unsigned* n_cand) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= in.n) return;
    const double big = __dmul_rn(8.0, sorted[in.n / 2]);
    if (radii[i] < big) return;
    if (sb_dist(in, i, res->centroid) <= __dmul_rn(1.05, radii[i])) cand[atomicAdd(n_cand, 1u)] = i;
}

// (a, ia) before (b, ib) in the order of std::pair<double, int>
__device__ __forceinline__ bool sb_pair_less(double a, int ia, double b, int ib) { return a < b || (!(b < a) && ia < ib); }

__global__ void sb_direct_choose(const SbInput in, const double* radii, const int* cand, const unsigned* n_cand, SbResult* res) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double key[kSbMaxDirect];
    int idx[kSbMaxDirect], m = 0;
    // the first 8 of the candidates ordered by (-|r|, index), by insertion
    for (unsigned q = 0; q < *n_cand; ++q) {
        const int i = cand[q];
        const double k = -radii[i];
        if (m == kSbMaxDirect && !sb_pair_less(k, i, key[m - 1], idx[m - 1])) continue;
        int p = m < kSbMaxDirect ? m++ : m - 1;
        while (p > 0 && sb_pair_less(k, i, key[p - 1], idx[p - 1])) { key[p] = key[p - 1]; idx[p] = idx[p - 1]; --p; }
        key[p] = k;
        idx[p] = i;
    }
    // cull order of the direct spheres: (-dist / max(1e-30, |r|), index)
    for (int a = 0; a < m; ++a) key[a] = -__ddiv_rn(sb_dist(in, idx[a], res->centroid), fmax(1e-30, radii[idx[a]]));
    for (int a = 1; a < m; ++a)
        for (int p = a; p > 0 && sb_pair_less(key[p], idx[p], key[p - 1], idx[p - 1]); --p) {
            const double tk = key[p]; key[p] = key[p - 1]; key[p - 1] = tk;
            const int ti = idx[p]; idx[p] = idx[p - 1]; idx[p - 1] = ti;
        }
    res->n_direct = m;
    for (int a = 0; a < m; ++a) res->direct[a] = idx[a];
}

// perm[k] = caller index of cull entry k: a listed sphere i goes to i minus the direct spheres before it (stable)
__global__ void __launch_bounds__(kSbBlock) sb_perm(int n, const SbResult* res, int* perm) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int m = res->n_direct;
    int before = 0;
    for (int a = 0; a < m; ++a) {
        if (res->direct[a] == i) { perm[n - m + a] = i; return; }
        before += res->direct[a] < i;
    }
    perm[i - before] = i;
}

// the blob's per-primitive sections (rt_set_scene_ex's host loops), plus the bounding spheres in the BvhLeafInput layout
struct SbBlob {
    float* c0r; float* c1; float* t0t1; unsigned* flags; int* mat; int* orig; int* cull_of;
    int* srec; float* scol; unsigned* tie;
    const int* mat_type; const float* mat_param; const int* mat_tex; const int* tex_type; const float* tex_params;
    int n_textures;
    double* bs_c0; double* bs_c1; double* bs_r;
    unsigned long long* tc_key; int* tc_val;   // listed leaves: ~bits of the bounding radius and cull index, the stable sort's input
    int n_list;
};

__global__ void __launch_bounds__(kSbBlock) sb_gather(const SbInput in, const int* perm, SbBlob b) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= in.n) return;
    const int i = perm ? perm[k] : k;
    const unsigned fl0 = in.flags ? in.flags[i] : 0u;
    const bool moving = sb_moving(in, i);
    const unsigned fl = moving ? fl0 : (fl0 & ~RT_SPHERE_MOVING);
    float c0[4], c1[3];
    for (int c = 0; c < 4; ++c) c0[c] = in.c0r[4 * (size_t)i + c];
    for (int c = 0; c < 3; ++c) c1[c] = moving ? in.c1[4 * (size_t)i + c] : c0[c];
    reinterpret_cast<float4*>(b.c0r)[k] = make_float4(c0[0], c0[1], c0[2], c0[3]);
    reinterpret_cast<float4*>(b.c1)[k] = make_float4(c1[0], c1[1], c1[2], 0.f);
    reinterpret_cast<float2*>(b.t0t1)[k] = moving ? make_float2(in.t0t1[2 * (size_t)i], in.t0t1[2 * (size_t)i + 1]) : make_float2(0.f, 1.f);
    b.flags[k] = fl;
    const int m = in.mat[i];
    b.mat[k] = m;
    b.orig[k] = i;
    b.cull_of[i] = k;
    const int tex = b.mat_tex[m];
    const bool has_tex = b.mat_type[m] != RT_MAT_DIELECTRIC && tex >= 0 && tex < b.n_textures;
    const int tex_type = has_tex ? b.tex_type[tex] : -1;
    reinterpret_cast<int4*>(b.srec)[k] = make_int4(b.mat_type[m], tex, tex_type, (int)fl);
    float col[3] = {0.f, 0.f, 0.f};
    if (tex_type == RT_TEX_CONSTANT)
        for (int c = 0; c < 3; ++c) col[c] = b.tex_params[12 * (size_t)tex + c];
    reinterpret_cast<float4*>(b.scol)[k] = make_float4(b.mat_param[m], col[0], col[1], col[2]);
    b.tie[k] = 0x80000000u | (unsigned)i;
    const double r = fabs((double)c0[3]);
    for (int c = 0; c < 3; ++c) { b.bs_c0[3 * (size_t)k + c] = (double)c0[c]; b.bs_c1[3 * (size_t)k + c] = (double)c1[c]; }
    b.bs_r[k] = r;
    if (k < b.n_list) { b.tc_key[k] = ~(unsigned long long)__double_as_longlong(r); b.tc_val[k] = k; }
}

// feature row p of `rows` = tc_tiles * 256: the leaf at rank q * words + w of the descending radius order, p = 32 w + q
// (the host's tc_row_k[(i % words) * 32 + i / words] = order[i]); a row without a leaf is padding (-1)
__global__ void __launch_bounds__(kSbBlock) sb_deal(const int* order, int n_list, int rows, int* row_k) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= rows) return;
    const int words = rows / 32, rank = (p % 32) * words + p / 32;
    row_k[p] = rank < n_list ? order[rank] : -1;
}

// build_cull_records for one leaf (generic = 0), operation for operation: the negated FP32 centre, the record's W and the
// tensor-core W in double
__device__ __forceinline__ void sb_record(const BvhLeafInput& in, int i, double win_lo, double win_hi, float neg[3], float* w, double* wtc) {
    const double eps = 0x1p-20, u = 0x1p-24;
    const double r = fabs(in.r[i]);
    double mid[3], half2 = 0.0, cmax = 0.0;
    const bool moving = (in.flags[i] & RT_SPHERE_MOVING) != 0u;
    for (int c = 0; c < 3; ++c) {
        const double p0 = in.c0[3 * (size_t)i + c];
        if (moving) {
            const double p1 = in.c1[3 * (size_t)i + c], t0 = in.t0t1[2 * (size_t)i], t1 = in.t0t1[2 * (size_t)i + 1];
            const double fa = __ddiv_rn(__dsub_rn(win_lo, t0), __dsub_rn(t1, t0)), fb = __ddiv_rn(__dsub_rn(win_hi, t0), __dsub_rn(t1, t0));
            const double pa = __dadd_rn(__dmul_rn(p0, __dsub_rn(1.0, fa)), __dmul_rn(p1, fa));
            const double pb = __dadd_rn(__dmul_rn(p0, __dsub_rn(1.0, fb)), __dmul_rn(p1, fb));
            mid[c] = __dmul_rn(0.5, __dadd_rn(pa, pb));
            const double dp = __dsub_rn(pb, pa);
            half2 = __dadd_rn(half2, __dmul_rn(__dmul_rn(0.25, dp), dp));
        } else {
            mid[c] = p0;
        }
        const double am = fabs(mid[c]);
        cmax = cmax < am ? am : cmax;   // std::max
    }
    const double rb = __dadd_rn(r, __dsqrt_rn(half2));
    const double e = moving ? __dmul_rn(0x1p-21, __dadd_rn(cmax, rb)) : 0.0;
    double cc = 0.0;
    for (int c = 0; c < 3; ++c) {
        neg[c] = __double2float_rn(-mid[c]);
        cc = __dadd_rn(cc, __dmul_rn((double)neg[c], (double)neg[c]));
    }
    const double re = __dadd_rn(rb, e);
    const double re2e = __dmul_rn(__dmul_rn(re, re), 1.0 + eps);
    const double r2i = __dadd_rn(__dadd_rn(re2e, __dmul_rn(48.0 * u, cc)), __dmul_rn(__dmul_rn(8.0 * u, re), re));
    *w = sb_round_up_f32(__dsub_rn(r2i, cc));
    *wtc = __dsub_rn(__dadd_rn(__dadd_rn(re2e, __dmul_rn(96.0 * u, cc)), __dmul_rn(__dmul_rn(24.0 * u, re), re)), cc);
}

// threads [0, n): leaf i's record, listed at i, direct at n_cull + (i - n_list); threads [n, n + n_cull - n_list): padding
__global__ void __launch_bounds__(kSbBlock) sb_cull_records(const BvhLeafInput in, int n, int n_list, int n_cull, double win_lo, double win_hi,
                                                            float4* cull_all) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n + n_cull - n_list) return;
    if (t >= n) { cull_all[n_list + (t - n)] = make_float4(0.f, 0.f, 0.f, -INFINITY); return; }
    float neg[3], w;
    double wtc;
    sb_record(in, t, win_lo, win_hi, neg, &w, &wtc);
    cull_all[t < n_list ? t : n_cull + (t - n_list)] = make_float4(neg[0], neg[1], neg[2], w);
}

__global__ void __launch_bounds__(kSbBlock) sb_tc_rows(const BvhLeafInput in, const int* row_k, int rows, double win_lo, double win_hi,
                                                       float* tc_out) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= rows) return;
    float slot[tc::KTOT];
    const int k = row_k[p];
    if (k >= 0) {
        float neg[3], w;
        double wtc;
        sb_record(in, k, win_lo, win_hi, neg, &w, &wtc);
        const double c[3] = {-(double)neg[0], -(double)neg[1], -(double)neg[2]};   // the centre AS STORED
        tc::sphere_slots(c, wtc, slot);
    } else {
        tc::padding_slots(slot);
    }
    float* tile = tc_out + (size_t)(p / tc::TILE_N) * (tc::B_TILE_BYTES / 4);
    for (int q = 0; q < tc::KTOT; ++q) tile[tc::canon_off(tc::TILE_N, p % tc::TILE_N, q) / 4] = slot[q];
}

}  // namespace rt
