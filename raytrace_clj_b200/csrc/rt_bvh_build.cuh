// rt_bvh_build.cuh — RT_ACCEL_BVH tree built on the device: a Karras LBVH (Karras 2012, "Maximizing parallelism in the
// construction of BVHs, octrees, and k-d trees") over the listed leaves, written straight into the node format that
// bvh_closest walks (4 float4 per node: left box lo.xyz hi.xyz, right box lo.xyz hi.xyz, then (left, right, 0, 0) as
// ints, a leaf child stored as ~k, the root at node 0).
//
//   bvh_leaf_boxes     one thread per leaf: the host builder's conservative leaf box, bit for bit (FP64 without FMA
//                      contraction, then the same float rounding and nextafterf widening), and the centroid bounds
//   bvh_morton         63-bit Morton code of the float centroid, quantised to 21 bits per axis in FP32
//   (cub radix sort)   (code, leaf) pairs; stable, so leaves with equal codes keep their cull order
//   bvh_hierarchy      one thread per internal node: range, split and children; parent links
//   bvh_fit            bottom up, one thread per leaf: the second thread to reach a node writes its children's boxes and
//                      its height and goes on; the root's height is the deepest leaf's depth
//
// The traversal does not depend on the shape of the tree (every leaf that survives a box gets the same exact FP64 test
// and the same tie key), so any valid tree gives the brute-force answer; the boxes must stay the host builder's, whose
// conservativeness the slab test relies on.
#pragma once

#include <cub/device/device_radix_sort.cuh>

#include "rt_device.cuh"

namespace rt {

constexpr unsigned kMortonAxisBits = 21;
constexpr int kBvhMaxDepth = 48;   // bvh_closest's stack entries: a tree whose deepest leaf is deeper is never traversed

// bounding spheres of the listed leaves as the host holds them (cull order); uploaded before every device build
struct BvhLeafInput {
    const double* c0;      // [3n] centre at t0
    const double* c1;      // [3n] centre at t1 (movers)
    const double* r;       // [n]
    const float* t0t1;     // [2n]
    const unsigned* flags; // [n]
};

// float <-> unsigned with the order of the floats (min / max by integer atomics)
__device__ __forceinline__ unsigned bvh_ordered(float f) {
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float bvh_unordered(unsigned u) {
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// the leaf box of ensure_bvh's host loop, operation for operation (std::min / std::max as written there)
__device__ __forceinline__ void bvh_leaf_box(const BvhLeafInput& in, int k, double win_lo, double win_hi, float lo[3], float hi[3]) {
    const bool moving = (in.flags[k] & RT_SPHERE_MOVING) != 0u;
    const double r = fabs(in.r[k]);
    for (int a = 0; a < 3; ++a) {
        double pa = in.c0[3 * (size_t)k + a], pb = pa;
        if (moving) {
            const double p0 = in.c0[3 * (size_t)k + a], p1 = in.c1[3 * (size_t)k + a];
            const double t0 = (double)in.t0t1[2 * (size_t)k], t1 = (double)in.t0t1[2 * (size_t)k + 1];
            const double fa = __ddiv_rn(__dsub_rn(win_lo, t0), __dsub_rn(t1, t0));
            const double fb = __ddiv_rn(__dsub_rn(win_hi, t0), __dsub_rn(t1, t0));
            pa = __dadd_rn(__dmul_rn(p0, __dsub_rn(1.0, fa)), __dmul_rn(p1, fa));
            pb = __dadd_rn(__dmul_rn(p0, __dsub_rn(1.0, fb)), __dmul_rn(p1, fb));
        }
        const double l = __dsub_rn(pb < pa ? pb : pa, r), h = __dadd_rn(pa < pb ? pb : pa, r);
        const double m = __dadd_rn(__dmul_rn(1e-6, __dadd_rn(__dadd_rn(fabs(l), fabs(h)), r)), 1e-30);
        lo[a] = nextafterf(__double2float_rn(__dsub_rn(l, m)), -INFINITY);
        hi[a] = nextafterf(__double2float_rn(__dadd_rn(h, m)), INFINITY);
    }
}

__device__ __forceinline__ float bvh_centroid(float lo, float hi) { return __fmul_rn(0.5f, __fadd_rn(lo, hi)); }

// boxes [6n] (lo.xyz, hi.xyz per leaf, cull order); cbounds [6] = ordered min.xyz, max.xyz of the centroids (preset to
// the identities)
__global__ void __launch_bounds__(256) bvh_leaf_boxes(const BvhLeafInput in, int n, double win_lo, double win_hi, float* boxes,
                                                      unsigned* cbounds) {
    __shared__ unsigned s_b[6];
    if (threadIdx.x < 6) s_b[threadIdx.x] = threadIdx.x < 3 ? 0xffffffffu : 0u;
    __syncthreads();
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) {
        float lo[3], hi[3];
        bvh_leaf_box(in, k, win_lo, win_hi, lo, hi);
        for (int a = 0; a < 3; ++a) {
            boxes[6 * (size_t)k + a] = lo[a];
            boxes[6 * (size_t)k + 3 + a] = hi[a];
            const unsigned c = bvh_ordered(bvh_centroid(lo[a], hi[a]));
            atomicMin(&s_b[a], c);
            atomicMax(&s_b[3 + a], c);
        }
    }
    __syncthreads();
    if (threadIdx.x < 3) atomicMin(&cbounds[threadIdx.x], s_b[threadIdx.x]);
    else if (threadIdx.x < 6) atomicMax(&cbounds[threadIdx.x], s_b[threadIdx.x]);
}

// 21 bits -> every third bit of 63
__device__ __forceinline__ unsigned long long bvh_spread3(unsigned v) {
    unsigned long long x = v & 0x1fffffu;
    x = (x | x << 32) & 0x1f00000000ffffull;
    x = (x | x << 16) & 0x1f0000ff0000ffull;
    x = (x | x << 8) & 0x100f00f00f00f00full;
    x = (x | x << 4) & 0x10c30c30c30c30c3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}

// q = min(floor((c - lo) / (hi - lo) * 2^21), 2^21 - 1) in FP32 with every operation rounded as written (numpy float32
// gives the same bits); an axis of zero extent quantises to 0.  Code: x at bits 3i + 2, y at 3i + 1, z at 3i.
__global__ void __launch_bounds__(256) bvh_morton(const float* boxes, int n, const unsigned* cbounds, unsigned long long* codes,
                                                  int* leaf) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    unsigned long long code = 0;
    for (int a = 0; a < 3; ++a) {
        const float lo = bvh_unordered(cbounds[a]), ext = __fsub_rn(bvh_unordered(cbounds[3 + a]), lo);
        const float c = bvh_centroid(boxes[6 * (size_t)k + a], boxes[6 * (size_t)k + 3 + a]);
        unsigned q = 0;
        if (ext > 0.f) {
            const float f = __fmul_rn(__fdiv_rn(__fsub_rn(c, lo), ext), (float)(1u << kMortonAxisBits));
            q = min(__float2uint_rz(f), (1u << kMortonAxisBits) - 1u);
        }
        code |= bvh_spread3(q) << (2 - a);
    }
    codes[k] = code;
    leaf[k] = k;
}

// common prefix of sorted keys i and j, a key being (code, position): -1 outside [0, n)
__device__ __forceinline__ int bvh_delta(const unsigned long long* codes, int n, int i, long long j) {
    if (j < 0 || j >= n) return -1;
    const unsigned long long a = codes[i], b = codes[j];
    return a != b ? __clzll((long long)(a ^ b)) : 64 + __clz(i ^ (int)j);
}

// internal node i in [0, n - 2] (n >= 2); parent[] holds the internal nodes' parents at [0, n - 1) and the leaves' (by
// sorted position) at n - 1 + p
__global__ void __launch_bounds__(256) bvh_hierarchy(const unsigned long long* codes, const int* sorted_leaf, int n, float4* nodes,
                                                     int* parent) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    const int d = bvh_delta(codes, n, i, i + 1) > bvh_delta(codes, n, i, i - 1) ? 1 : -1;
    const int dmin = bvh_delta(codes, n, i, (long long)i - d);
    long long lmax = 2;
    while (bvh_delta(codes, n, i, i + lmax * d) > dmin) lmax *= 2;
    long long l = 0;
    for (long long t = lmax / 2; t >= 1; t /= 2)
        if (bvh_delta(codes, n, i, i + (l + t) * d) > dmin) l += t;
    const int j = (int)(i + l * d);
    const int dnode = bvh_delta(codes, n, i, j);
    long long s = 0, t = l;
    do {
        t = (t + 1) / 2;
        if (bvh_delta(codes, n, i, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    const int gamma = (int)(i + s * d) + min(d, 0);
    int left, right;
    if (min(i, j) == gamma) { left = ~__ldg(&sorted_leaf[gamma]); parent[n - 1 + gamma] = i; }
    else { left = gamma; parent[gamma] = i; }
    if (max(i, j) == gamma + 1) { right = ~__ldg(&sorted_leaf[gamma + 1]); parent[n - 1 + gamma + 1] = i; }
    else { right = gamma + 1; parent[gamma + 1] = i; }
    nodes[4 * (size_t)i + 3] = make_float4(__int_as_float(left), __int_as_float(right), 0.f, 0.f);
}

// box of a child as its parent stores it: a leaf's own box, or the union of an internal node's two children's boxes
__device__ __forceinline__ void bvh_child_box(const float4* nodes, const float* boxes, const int* height, int c, float lo[3], float hi[3],
                                              int* h) {
    if (c < 0) {
        const float* b = boxes + 6 * (size_t)(~c);
        for (int a = 0; a < 3; ++a) { lo[a] = b[a]; hi[a] = b[3 + a]; }
        *h = 0;
        return;
    }
    // written by another thread of this launch: read through L2
    const float4 A = __ldcg(&nodes[4 * (size_t)c]), B = __ldcg(&nodes[4 * (size_t)c + 1]), C = __ldcg(&nodes[4 * (size_t)c + 2]);
    lo[0] = fminf(A.x, B.z); lo[1] = fminf(A.y, B.w); lo[2] = fminf(A.z, C.x);
    hi[0] = fmaxf(A.w, C.y); hi[1] = fmaxf(B.x, C.z); hi[2] = fmaxf(B.y, C.w);
    *h = __ldcg(&height[c]);
}

// one thread per sorted leaf position; arrive[] zeroed; out_depth[0] = depth of the deepest leaf (root = depth 0)
__global__ void __launch_bounds__(256) bvh_fit(const float* boxes, const int* parent, int n, float4* nodes, unsigned* arrive, int* height,
                                               int* out_depth) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    int node = parent[n - 1 + p];
    for (;;) {
        __threadfence();                                    // this thread's writes below node are visible before it arrives
        if (atomicAdd(&arrive[node], 1u) == 0u) return;     // the sibling subtree is not done: its last thread continues
        __threadfence();
        const int4 ch = __ldg(reinterpret_cast<const int4*>(&nodes[4 * (size_t)node + 3]));
        float llo[3], lhi[3], rlo[3], rhi[3];
        int hl, hr;
        bvh_child_box(nodes, boxes, height, ch.x, llo, lhi, &hl);
        bvh_child_box(nodes, boxes, height, ch.y, rlo, rhi, &hr);
        nodes[4 * (size_t)node] = make_float4(llo[0], llo[1], llo[2], lhi[0]);
        nodes[4 * (size_t)node + 1] = make_float4(lhi[1], lhi[2], rlo[0], rlo[1]);
        nodes[4 * (size_t)node + 2] = make_float4(rlo[2], rhi[0], rhi[1], rhi[2]);
        const int h = 1 + max(hl, hr);
        height[node] = h;
        if (node == 0) { *out_depth = h; return; }
        node = parent[node];
    }
}

// n == 1: the lone leaf is both children of the root (hitable.clj:113-114), as in the host builder
__global__ void bvh_single_leaf(const float* boxes, float4* nodes, int* out_depth) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const float* b = boxes;
    nodes[0] = make_float4(b[0], b[1], b[2], b[3]);
    nodes[1] = make_float4(b[4], b[5], b[0], b[1]);
    nodes[2] = make_float4(b[2], b[3], b[4], b[5]);
    nodes[3] = make_float4(__int_as_float(~0), __int_as_float(~0), 0.f, 0.f);
    *out_depth = 1;
}

}  // namespace rt
