// rt_cull_tc.cuh — the brute-force cull on the 5th-generation tensor cores (tcgen05 / TMEM, sm_100a).
// Included by rt_kernels.cuh (inside namespace rt, after the FP32 cull it is checked against).
//
// The conservative test "can the LINE of this ray meet this (inflated) sphere" is a bilinear form of per-ray and
// per-sphere features, i.e. every (ray, sphere) pair of a tile is one element of a GEMM:
//     disc = (h.(o - c))^2 - |o - c|^2 + R2                                         |h|^2 = 1 + eps
//          = [P^2 - Q] + [R2 - c.c] + sum_i c_i [2 (o_i - P h_i)] + sum_i c_i^2 [h_i^2] + sum_{i<j} 2 c_i c_j [h_i h_j]
// with P = o.h, Q = o.o: 11 feature products.  FP32 accuracy on TF32 tensor cores comes from splitting every feature
// into hi + lo TF32 parts (hi hi + hi lo + lo hi; the two seeds W = R2 - c.c and g0 = P^2 - Q in three / two parts):
// 32 K-slots = 4 chained tcgen05.mma (M 128 rays x N 256 spheres x K 8, kind::tf32) per tile, accumulated in TMEM.
// The epilogue only collects SIGN BITS: one funnel shift per pair (sign set = no intersection), exactly the mask
// words of the FP32 cull.  A clear bit is a CANDIDATE (~0.5 % of the pairs); candidates are compacted per warp and
// confirmed with the FP32 cull's own key (which also drops spheres behind the origin), so the pairs this kernel
// emits are a subset of wf_cull's and still a superset of the exact hits (tests: rt_cull_check with cull_tc = 1,
// and every render test — the FP64 refine downstream is unchanged, so images are bit-identical).
//
// Rounding budget (u = 2^-24; DESIGN.md "Precision"): feature rounding on the ray side <= u (15.5 |o|^2 + 5.2 |c|^2);
// hi/lo split (round-to-nearest TF32 parts, lo.lo dropped) <= 12 u per product <= u (16 |o|^2 + 24 |c|^2);
// tensor-core accumulation (operands truncated to TF32 = exact for our parts; 4 chained K = 8 MMAs measured at
// <= 7 u sum|terms| by csrc/tcprobe.cu, budgeted at 16 u) <= u (32 |o|^2 + 48 |c|^2 + 16 R2).  The ray's share
// (80 u |o|^2) is taken off Q, the sphere's (96 u c.c + 24 u R2) is added to W on the host (build_cull_records).
//
// CTA = 16 epilogue warps + 1 MMA-issuing warp + 4 producer warps, one CTA per SM (the two accumulator buffers take all
// 512 TMEM columns).  The sphere features of a launch stay resident in shared memory (<= 4 tiles of 256 = 1024 leaves);
// a longer list is covered by several launches per iteration, each over its own 1024 leaves (WaveParams::tc_tile0).

namespace tc {

constexpr int EW = 16;                         // epilogue warps (warps 0 .. 15)
constexpr int PG = 1;                          // producer groups (4 warps each, one ray of the tile per thread): group q builds the
constexpr int PW = 4 * PG;                     //   ray tiles it = q, q + PG, ...  (measured: ~800 cycles per tile, one group keeps up)
constexpr int THREADS = (EW + 1 + PW) * 32;    // epilogue warps 0 .. 15, the MMA warp 16, producer warps 17 .. 20
constexpr int MAX_SLOTS = 4;                   // ray-tile buffers the producers can run ahead through
constexpr int TILE_M = 128;                    // rays per tile = TMEM lanes
constexpr int TILE_N = 256;                    // spheres per MMA group = TMEM columns of one accumulator buffer
constexpr int KTOT = 32;                       // K-slots (TF32) per pair: 4 MMAs of K = 8
constexpr int A_BYTES = TILE_M * KTOT * 4;     // 16 KB per ray tile
constexpr int B_TILE_BYTES = TILE_N * KTOT * 4;   // 32 KB per sphere tile
constexpr int MAX_TILES = 4;                   // resident sphere tiles
constexpr int MIN_LEAVES = 160;                // shorter lists stay on the FP32 loop (a 256-column tile would be mostly padding)
constexpr int CAND_CAP = 256;                  // per-warp candidate list (one ray tile)
constexpr int PAIR_CHUNK = 64;                 // pair slots a warp reserves at a time (one atomic)
constexpr float RAY_DEFLATE = 1.0f - 5.0e-6f;  // 1 - 84 u: the ray's share of the rounding budget, taken off |o|^2
constexpr float DEAD = -1.0e30f;               // g0 of a dead ray / W of a padding sphere: disc < 0 against anything

__host__ __device__ inline size_t canon_off(int rows, int r, int k) {   // bytes; K-major, no swizzle: core matrix = 8 rows x 16 B
    return (size_t)(k / 4) * ((size_t)rows * 16) + (size_t)(r / 8) * 128 + (size_t)(r % 8) * 16 + (size_t)(k % 4) * 4;
}
// sphere features + their FP32 records, `slots` ray tiles + their FP32 constants, candidate lists, barriers
inline size_t smem_bytes(int tiles, int slots) {
    return (size_t)tiles * B_TILE_BYTES + (size_t)tiles * TILE_N * (16 + 4) + (size_t)slots * (A_BYTES + TILE_M * 32) + (size_t)EW * CAND_CAP * 4 + 1024;
}
inline int slots_for(int tiles, size_t smem_limit) {
    int s = MAX_SLOTS;
    while (s > 2 && smem_bytes(tiles, s) > smem_limit) --s;
    return s;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// a protocol error must end the kernel with an error, never hang the device
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    for (unsigned spin = 0; spin < 0x40000000u; ++spin)
        if (mbar_try_wait(bar, parity)) return;
    __trap();
}
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr >> 4) & 0x3fffu) | ((uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16) | ((uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32) |
           (1ull << 46);               // sm_100 descriptor version; no swizzle, base offset 0
}
#ifndef RT_TC_NBLK
#define RT_TC_NBLK 1
#endif
constexpr int NBLK = RT_TC_NBLK;               // column blocks of an accumulator buffer that advance on their own (own full / empty barriers,
constexpr int BLOCK_N = TILE_N / NBLK;         //   own MMAs of N = BLOCK_N).  Kept as a compile-time experiment: with 4 blocks the epilogue's load
constexpr int BLOCK_WARPS = EW / NBLK;         //   phase drops from 1250 to 800 cycles per tile (no collisions), but a tcgen05.mma costs ~128 cycles
                                               //   whatever N <= 256, so the tensor pipe becomes the bottleneck (C2: 7.56 ms; 2 blocks 6.05; 1 block 5.76)
constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BLOCK_N >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);   // f32 += tf32 x tf32, both K-major
__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
    asm volatile("{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}"
                 ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(IDESC), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
#define RT_TMEM_LD32(taddr, v)                                                                                                \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "                                                                   \
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "                                   \
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"                   \
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),           \
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),     \
                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),   \
                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])    \
                 : "r"(taddr))
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// x = hi + lo + residual, hi and lo TF32-representable (round to nearest), |residual| <= 2^-22 |x|
__host__ __device__ inline float tf32_rn(float x) {
#ifdef __CUDA_ARCH__
    return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
#else
    uint32_t b; memcpy(&b, &x, 4); b = (b + 0x1000u) & 0xffffe000u; memcpy(&x, &b, 4); return x;
#endif
}
__device__ __forceinline__ void split2(float x, float& hi, float& lo) {
    hi = tf32_rn(x);
    lo = tf32_rn(x - hi);             // x - hi is exact
}

// K-slot table (ray value | sphere value); cii = c_i^2, cij = 2 c_i c_j, g_i = 2 (o_i - P h_i), q_ij = h_i h_j:
//   0 g0.hi|1     1 g0.lo|1     2 1|W.hi      3 1|W.lo      4 gx.hi|cx.hi   5 gx.hi|cx.lo   6 gx.lo|cx.hi   7 1|W.lo2
//   8 gy.hi|cy.hi 9 gy.hi|cy.lo 10 gy.lo|cy.hi 11 qyz.hi|cyz.lo  12 gz.hi|cz.hi 13 gz.hi|cz.lo 14 gz.lo|cz.hi 15 qyz.lo|cyz.hi
//   16..18 qxx|cxx   19..21 qyy|cyy   22..24 qzz|czz   25..27 qxy|cxy   28..30 qxz|cxz  (hi|hi, hi|lo, lo|hi)   31 qyz.hi|cyz.hi
// FP64 product / difference rounded as written on both sides: the device must not contract them into an FMA
__host__ __device__ inline double dmul_rn(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
__host__ __device__ inline double dsub_rn(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}

// One sphere's 32 slots (build_cull_records on the host, sb_tc_rows on the device: the same bits).  c = centre AS STORED in
// the FP32 record, W in double.
__host__ __device__ inline void sphere_slots(const double c[3], double W, float out[KTOT]) {
    auto sp2 = [](double x, float& hi, float& lo) { hi = tf32_rn((float)x); lo = tf32_rn((float)dsub_rn(x, (double)hi)); };
    float wh = tf32_rn((float)W), wl = tf32_rn((float)dsub_rn(W, (double)wh)), wl2 = tf32_rn((float)dsub_rn(dsub_rn(W, (double)wh), (double)wl));
    float ch[3], cl[3], dh[3], dl[3], eh[3], el[3];   // c_i, c_i^2, cross terms (xy, xz, yz)
    for (int i = 0; i < 3; ++i) { sp2(c[i], ch[i], cl[i]); sp2(dmul_rn(c[i], c[i]), dh[i], dl[i]); }
    sp2(dmul_rn(dmul_rn(2.0, c[0]), c[1]), eh[0], el[0]); sp2(dmul_rn(dmul_rn(2.0, c[0]), c[2]), eh[1], el[1]);
    sp2(dmul_rn(dmul_rn(2.0, c[1]), c[2]), eh[2], el[2]);
    const float s[KTOT] = {1.f, 1.f, wh, wl, ch[0], cl[0], ch[0], wl2, ch[1], cl[1], ch[1], el[2], ch[2], cl[2], ch[2], eh[2],
                           dh[0], dl[0], dh[0], dh[1], dl[1], dh[1], dh[2], dl[2], dh[2], eh[0], el[0], eh[0], eh[1], el[1], eh[1], eh[2]};
    for (int k = 0; k < KTOT; ++k) out[k] = s[k];
}
__host__ __device__ inline void padding_slots(float out[KTOT]) {
    for (int k = 0; k < KTOT; ++k) out[k] = 0.f;
    out[0] = 1.f;                      // against g0.hi: a DEAD ray stays dead (0 x 0 would be +0 = "candidate")
    out[2] = DEAD;                     // W.hi against the ray's 1
}

struct Smem {
    float* B;                          // [tiles][256 x 32] canonical
    float4* rec;                       // [tiles * 256] the FP32 cull records of the same leaves, in ROW order (confirm step)
    int* row_k;                        // [tiles * 256] cull index of the leaf in feature row p (rows are a fixed shuffle of the list,
                                       //   so that every warp's 64-column block sees the same mix of leaves), -1 = padding row
    unsigned char* A0;                 // [slots][128 x 32] canonical ray tiles
    float4* ray0;                      // [slots][128][2]: the FP32 cull's per-ray constants (confirm step)
    uint32_t* cand;                    // [EW][CAND_CAP]
    uint64_t* a_ready;                 // [slots] producers (128 arrivals) -> MMA warp, epilogue: A[s], ray[s], tile_of[s] written
    uint64_t* a_free;                  // [slots] MMA warp (commit) -> producers: every MMA that read A[s] has completed
    uint64_t* ray_free;                // [slots] epilogue (one arrival per warp) -> producers: ray[s] has been used
    uint64_t* d_full;                  // [2][NBLK] MMA warp (commit) -> the block's 4 epilogue warps: its 64 columns of buffer b are written
    uint64_t* d_empty;                 // [2][NBLK] the block's warps (one arrival each) -> MMA warp: those columns have been read
    int* tile_of;                      // [slots] ray tile in A[s], or -1 = no more work
    uint32_t* tmem_base;
    unsigned* cand_n;                  // [EW] candidates in each warp's list
    __device__ __forceinline__ float* A(unsigned s) const { return reinterpret_cast<float*>(A0 + (size_t)s * A_BYTES); }
    __device__ __forceinline__ float4* ray(unsigned s) const { return ray0 + (size_t)s * TILE_M * 2; }
};
__device__ __forceinline__ Smem carve(unsigned char* base, int tiles, int slots) {
    Smem S;
    S.B = reinterpret_cast<float*>(base);
    unsigned char* p = base + (size_t)tiles * B_TILE_BYTES;
    S.rec = reinterpret_cast<float4*>(p);
    p += (size_t)tiles * TILE_N * 16;
    S.row_k = reinterpret_cast<int*>(p);
    p += (size_t)tiles * TILE_N * 4;
    S.A0 = p;
    p += (size_t)slots * A_BYTES;
    S.ray0 = reinterpret_cast<float4*>(p);
    p += (size_t)slots * TILE_M * 32;
    S.cand = reinterpret_cast<uint32_t*>(p);
    p += (size_t)EW * CAND_CAP * 4;
    uint64_t* bars = reinterpret_cast<uint64_t*>(p);
    S.a_ready = bars; S.a_free = bars + MAX_SLOTS; S.ray_free = bars + 2 * MAX_SLOTS;
    S.d_full = bars + 3 * MAX_SLOTS; S.d_empty = bars + 3 * MAX_SLOTS + 2 * NBLK;
    int* ints = reinterpret_cast<int*>(bars + 3 * MAX_SLOTS + 4 * NBLK);
    S.tile_of = ints;
    S.tmem_base = reinterpret_cast<uint32_t*>(ints + MAX_SLOTS);
    S.cand_n = reinterpret_cast<unsigned*>(ints + MAX_SLOTS + 4);
    return S;
}

}  // namespace tc

// RT_TC_CHECK (compile-time, debugging): index checks before every global access of the kernel
#ifdef RT_TC_CHECK
#define TC_CHECK(cond, what, a, b) do { if (!(cond)) { printf("wf_cull_tc check failed: %s (%u, %u) block %u thread %u\n", what, (unsigned)(a), (unsigned)(b), blockIdx.x, threadIdx.x); __trap(); } } while (0)
#else
#define TC_CHECK(cond, what, a, b)
#endif

// One ray of the tile: features into A[slot] (canonical layout), FP32 cull constants into ray[slot].
// v = virtual queue index (v < n_g: path in flight, its record is loaded; else fresh: generated here and written).
template <bool VIEWS>
__device__ __forceinline__ void tc_produce_ray(const WaveParams& W, const tc::Smem& S, int slot, int rl, bool live, unsigned v, unsigned n_g,
                                               unsigned p0, unsigned long long gen_base, int cur) {
    const RenderParams& P = W.base;
    float f[tc::KTOT];
    float4 r0, r1;
    if (live) {
        float4* qc = cur ? W.queue[1] : W.queue[0];
        float4 a, b;
        if (v >= n_g && W.tc_pass != 0) {                      // a fresh entry whose ray an earlier pass generated and stored
            const size_t e = (size_t)(p0 + (v - n_g));
            a = qc[3 * e];
            b = qc[3 * e + 1];
        } else if (v >= n_g) {
            float4 c;
            float4* q = qc + 3 * (size_t)(p0 + (v - n_g));
            TC_CHECK(p0 + (v - n_g) < (unsigned)W.capacity, "fresh entry", p0 + (v - n_g), W.capacity);
            TC_CHECK(gen_base + (v - n_g) < P.total_work, "work item", (unsigned)(gen_base + (v - n_g)), (unsigned)P.total_work);
            make_path<VIEWS>(P, gen_base + (v - n_g), a, b, c);
            q[0] = a; q[1] = b; q[2] = c;
        } else {
            TC_CHECK(v < (unsigned)W.capacity, "entry in flight", v, W.capacity);
            a = qc[3 * (size_t)v];
            b = qc[3 * (size_t)v + 1];
        }
        const float aa = fmaf(b.z, b.z, fmaf(b.y, b.y, b.x * b.x));
        const float inv = rsqrtf(aa);
        const float qq = fmaf(a.z, a.z, fmaf(a.y, a.y, a.x * a.x));
        {   // the FP32 cull's constants, exactly Culler::set_ray
            const float s = inv * ((1.0f + 0.5f * CULL_EPS) * 0.70710678118654752f);
            const float hx = b.x * s, hy = b.y * s, hz = b.z * s;
            r0 = make_float4(hx, hy, hz, fmaf(a.z, hz, fmaf(a.y, hy, a.x * hx)));
            r1 = make_float4(-2.0f * a.x, -2.0f * a.y, -2.0f * a.z, qq * RAY_DEFLATE);
        }
        const float s = inv * (1.0f + 0.5f * CULL_EPS);
        const float hx = b.x * s, hy = b.y * s, hz = b.z * s;
        const float Pd = fmaf(a.z, hz, fmaf(a.y, hy, a.x * hx));
        const float g0 = fmaf(Pd, Pd, -(qq * tc::RAY_DEFLATE));
        const float gx = 2.0f * fmaf(-Pd, hx, a.x), gy = 2.0f * fmaf(-Pd, hy, a.y), gz = 2.0f * fmaf(-Pd, hz, a.z);
        float h_, l_;
        tc::split2(g0, h_, l_); f[0] = h_; f[1] = l_;
        f[2] = 1.f; f[3] = 1.f; f[7] = 1.f;
        tc::split2(gx, h_, l_); f[4] = h_; f[5] = h_; f[6] = l_;
        tc::split2(gy, h_, l_); f[8] = h_; f[9] = h_; f[10] = l_;
        tc::split2(gz, h_, l_); f[12] = h_; f[13] = h_; f[14] = l_;
        tc::split2(hx * hx, h_, l_); f[16] = h_; f[17] = h_; f[18] = l_;
        tc::split2(hy * hy, h_, l_); f[19] = h_; f[20] = h_; f[21] = l_;
        tc::split2(hz * hz, h_, l_); f[22] = h_; f[23] = h_; f[24] = l_;
        tc::split2(hx * hy, h_, l_); f[25] = h_; f[26] = h_; f[27] = l_;
        tc::split2(hx * hz, h_, l_); f[28] = h_; f[29] = h_; f[30] = l_;
        tc::split2(hy * hz, h_, l_); f[31] = h_; f[11] = h_; f[15] = l_;
    } else {
#pragma unroll
        for (int k = 0; k < tc::KTOT; ++k) f[k] = 0.f;
        f[0] = tc::DEAD;               // g0.hi against the 1 every row (padding included) carries in slot 0
        f[2] = 1.f;                    // and a padding row's W.hi = DEAD counts too: dead ray x padding row = -2e30, never +0
        r0 = make_float4(1.f, 0.f, 0.f, 0.f);
        r1 = make_float4(0.f, 0.f, 0.f, CUDART_INF_F);
    }
    unsigned char* Ab = reinterpret_cast<unsigned char*>(S.A((unsigned)slot)) + (size_t)(rl >> 3) * 128 + (size_t)(rl & 7) * 16;
#pragma unroll
    for (int kc = 0; kc < tc::KTOT / 4; ++kc)
        *reinterpret_cast<float4*>(Ab + (size_t)kc * (tc::TILE_M * 16)) = make_float4(f[4 * kc], f[4 * kc + 1], f[4 * kc + 2], f[4 * kc + 3]);
    S.ray((unsigned)slot)[2 * rl] = r0;
    S.ray((unsigned)slot)[2 * rl + 1] = r1;
}

// per-warp pair emission: pair slots are reserved PAIR_CHUNK at a time with one atomic and there is always ONE reservation
// requested ahead (nobody waits for an atomic's round trip unless a warp emits a whole chunk faster than that); slots left
// unused are padded with PAIR_NULL (wf_refine skips those)
struct TcEmit {
    unsigned pos, end;                 // warp-uniform: next free slot / end of the current reservation
    unsigned next;                     // lane 0: start of the reservation requested ahead (if `ahead`)
    bool ahead;                        // a warp that never emits reserves nothing
    unsigned pads;                     // padding slots written so far (WaveState::pad: wf_refine takes them off the candidate count)
};
__device__ __forceinline__ void tc_pad(const WaveParams& W, TcEmit& E, unsigned from, unsigned to, unsigned lane) {
    TC_CHECK(to <= W.pair_cap, "pad", from, to);
#ifdef RT_TC_CHECK
    for (unsigned i = from + lane; i < to; i += 32) W.pairs[i] = make_uint2(PAIR_NULL, (blockIdx.x << 8) | (threadIdx.x >> 5));
#else
    for (unsigned i = from + lane; i < to; i += 32) W.pairs[i] = make_uint2(PAIR_NULL, 0u);
#endif
    if (to > from) E.pads += to - from;
}
__device__ __forceinline__ void tc_request(const WaveParams& W, TcEmit& E, unsigned lane) {
    unsigned b = 0;
    if (lane == 0) b = atomicAdd(&W.st->npairs, (unsigned)tc::PAIR_CHUNK);
    E.next = b;
    E.ahead = true;
}

// warp-converged: the lanes with `emit` append (entry, k) to the warp's pair reservation
__device__ __forceinline__ void tc_emit(const WaveParams& W, TcEmit& E, bool emit, unsigned entry, unsigned k, unsigned lane) {
    const unsigned bal = __ballot_sync(0xffffffffu, emit);
    const unsigned total = __popc(bal);
    if (total == 0) return;
    if (E.pos + total > E.end) {   // move to the reservation requested ahead (the rest of the old one becomes padding), request another
        tc_pad(W, E, E.pos, E.end, lane);
        if (!E.ahead) tc_request(W, E, lane);             // the warp's first pairs of this launch: the one atomic it waits for
        const unsigned b = __shfl_sync(0xffffffffu, E.next, 0);
        E.pos = min(b, W.pair_cap);
        E.end = min(b + (unsigned)tc::PAIR_CHUNK, W.pair_cap);
        tc_request(W, E, lane);
    }
    if (emit) {
        const unsigned w = E.pos + __popc(bal & ((1u << lane) - 1u));
        TC_CHECK(entry < (unsigned)W.capacity && k < (unsigned)W.base.sc.n_list, "pair", entry, k);
        if (w < E.end) W.pairs[w] = make_uint2(entry, k);
        else W.best_key[entry] = BEST_KEY_OVERFLOW;       // pair buffer full: wf_shade re-intersects this entry exactly
    }
    E.pos = min(E.pos + total, E.end);
}

// The FP32 cull's own test of one (ray, feature row): Culler::key_bits, general form, on the constants the producers left
__device__ __forceinline__ bool tc_confirm(const tc::Smem& S, float4 r0, float4 r1, unsigned row, int& kk) {
    const float4 R = S.rec[row];
    kk = S.row_k[row];
    const float cc = fmaf(R.x, r0.x, fmaf(R.y, r0.y, fmaf(R.z, r0.z, r0.w)));
    const float s = fmaf(R.x, r1.x, fmaf(R.y, r1.y, fmaf(R.z, r1.z, R.w)));
    const float key = fmaf(-cc, fabsf(cc), fmaf(cc, cc, s - r1.w));
    return (__float_as_uint(key) >> 31) == 0u && kk >= 0;     // (a padding row never gets here: W = DEAD)
}

// A warp whose candidate list overflowed (dozens of leaves along its rays' lines: loose bounding spheres, a dense layer)
// drops the list and redoes its share of the tile — 32 rays x its 64 columns of every group — with the FP32 test itself:
// as slow as the FP32 loop for that warp and tile, never a lost pair, no exact re-intersection downstream.
__device__ __noinline__ void tc_redo_fp32(const WaveParams& W, const tc::Smem& S, int slot, unsigned tile, unsigned n, unsigned n_g, unsigned n_p,
                                          int tiles, unsigned cb, unsigned rl) {
    if (tile * tc::TILE_M + rl >= n) return;
    const float4 r0 = S.ray((unsigned)slot)[2 * rl], r1 = S.ray((unsigned)slot)[2 * rl + 1];
    const unsigned entry = wf_entry(tile * tc::TILE_M + rl, n_g, n_p, (unsigned)W.capacity);
    for (int j = 0; j < tiles; ++j)
        for (unsigned q = 0; q < 64u; ++q) {
            int kk;
            if (!tc_confirm(S, r0, r1, (unsigned)j * tc::TILE_N + cb * 64u + q, kk)) continue;
            const unsigned w = atomicAdd(&W.st->npairs, 1u);  // (single slots, outside the warp's reservation: nothing to pad; a rare path)
            if (w < W.pair_cap) W.pairs[w] = make_uint2(entry, (unsigned)kk);
            else W.best_key[entry] = BEST_KEY_OVERFLOW;       // pair buffer full: wf_shade re-intersects this entry exactly
        }
}

// FP32 confirm + emission of this warp's candidate list (ray-local index << 20 | feature row)
__device__ __forceinline__ void tc_drain(const WaveParams& W, const tc::Smem& S, int slot, unsigned tile, unsigned n_g, unsigned n_p,
                                         const uint32_t* cand, unsigned ncand, TcEmit& E, unsigned lane) {
    for (unsigned base = 0; base < ncand; base += 32) {
        const unsigned idx = base + lane;
        bool emit = false;
        unsigned k = 0, entry = 0;
        if (idx < ncand) {
            const uint32_t c = cand[idx];
            const unsigned rl = c >> 20, row = c & 0xfffffu;
            TC_CHECK(rl < 128u && row < (unsigned)W.tc_launch_tiles * 256u, "candidate", c, ncand);
            int kk;
            emit = tc_confirm(S, S.ray((unsigned)slot)[2 * rl], S.ray((unsigned)slot)[2 * rl + 1], row, kk);
            k = (unsigned)kk;
            entry = wf_entry(tile * tc::TILE_M + rl, n_g, n_p, (unsigned)W.capacity);
        }
        tc_emit(W, E, emit, entry, k, lane);
    }
}

// RT_TC_TIMING (compile-time): per-role cycle accounting of CTA 0, printed at the end of the launch
#ifdef RT_TC_TIMING
#define TC_T(var) const long long var = clock64()
#define TC_ACC(slot, since) tacc[slot] += clock64() - (since)
#else
#define TC_T(var)
#define TC_ACC(slot, since)
#endif
// VIEWS: instantiated for rt_render_views (false: single-camera renders)
template <bool VIEWS>
__global__ void __launch_bounds__(tc::THREADS, 1) wf_cull_tc(const __grid_constant__ WaveParams W) {
    TraceScope trace(W.trace);
    const RenderParams& P = W.base;
    extern __shared__ __align__(1024) unsigned char tc_smem[];
    if (W.st->mode != MODE_RUN) return;
    const unsigned n_g = W.st->cnt[W.cur][0], n_p = W.st->cnt[W.cur][1], n = n_g + n_p;
    if (n == 0) return;
    const unsigned long long gen_base = W.st->gen_base[W.cur];
    const unsigned p0 = (unsigned)W.capacity - n_p;
    const int tiles = W.tc_launch_tiles;
    const unsigned slots = (unsigned)W.tc_slots;
    const tc::Smem S = tc::carve(tc_smem, tiles, (int)slots);
    const unsigned tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;
    if (blockIdx.x == 0 && tid == 0 && W.tc_pass == 0) atomicAdd(&P.counters[DC_RAYS], (unsigned long long)n);

    // this CTA's ray tiles: a contiguous run
    const unsigned total_tiles = (n + tc::TILE_M - 1) / tc::TILE_M;
    const unsigned per_cta = W.claims_per_warp > 0 ? (unsigned)W.claims_per_warp : (total_tiles + gridDim.x - 1) / gridDim.x;
    const unsigned first = blockIdx.x * per_cta, last = min(first + per_cta, total_tiles);
    if (first >= last) return;         // CTA-uniform

    if (tid == 0) {
        for (unsigned i = 0; i < slots; ++i) {
            tc::mbar_init(&S.a_ready[i], tc::TILE_M);
            tc::mbar_init(&S.a_free[i], 1);
            tc::mbar_init(&S.ray_free[i], tc::EW);
        }
        for (int i = 0; i < 2 * tc::NBLK; ++i) {
            tc::mbar_init(&S.d_full[i], 1);
            tc::mbar_init(&S.d_empty[i], tc::BLOCK_WARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == tc::EW) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc::smem_u32(S.tmem_base)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid < tc::EW) S.cand_n[tid] = 0u;
    {   // the sphere features of the whole list (already in the canonical layout) and their FP32 records: global (L2) -> shared
        const float4* src = reinterpret_cast<const float4*>(P.sc.cull_tc) + (size_t)W.tc_tile0 * (tc::B_TILE_BYTES / 16);
        float4* dst = reinterpret_cast<float4*>(S.B);
        const int n4 = tiles * (tc::B_TILE_BYTES / 16);
        for (int i = (int)tid; i < n4; i += tc::THREADS) dst[i] = __ldg(&src[i]);
        for (int i = (int)tid; i < tiles * tc::TILE_N; i += tc::THREADS) {
            const int k = __ldg(&P.sc.tc_row_k[(size_t)W.tc_tile0 * tc::TILE_N + i]);
            S.row_k[i] = k;
            S.rec[i] = k >= 0 ? __ldg(&P.sc.cull_a[k]) : make_float4(0.f, 0.f, 0.f, -CUDART_INF_F);
        }
    }
    tc::fence_async_smem();
    tc::fence_before();
    __syncthreads();
    tc::fence_after();
    const uint32_t tmem = *S.tmem_base;
    const unsigned n_it = last - first;
#ifdef RT_TC_TIMING
    long long tacc[6] = {0, 0, 0, 0, 0, 0};
    const long long t_begin = clock64();
#endif

    if (warp > tc::EW) {
        // ===== producers: group q (4 warps, thread = one ray) builds tiles it = q, q + PG, ...; `slots` tiles ahead at most =====
        const unsigned pt = tid - (tc::EW + 1) * 32, rl = pt & (tc::TILE_M - 1), q = pt / tc::TILE_M;
        for (unsigned it = q; it <= n_it; it += tc::PG) {       // it == n_it: the end marker
            const unsigned s = it % slots, ph = (it / slots) & 1u;
            TC_T(t0);
            if (it >= slots) {
                tc::mbar_wait(&S.a_free[s], ph ^ 1u);
                TC_ACC(0, t0);
                TC_T(t1);
                tc::mbar_wait(&S.ray_free[s], ph ^ 1u);
                TC_ACC(1, t1);
            }
            TC_T(t2);
            if (it < n_it) {
                const unsigned v = (first + it) * tc::TILE_M + rl;
                tc_produce_ray<VIEWS>(W, S, (int)s, (int)rl, v < n, v, n_g, p0, gen_base, W.cur);
            }
            TC_ACC(2, t2);
            if (rl == 0) S.tile_of[s] = it < n_it ? (int)(first + it) : -1;
            tc::fence_async_smem();
            tc::mbar_arrive(&S.a_ready[s]);
        }
    } else if (warp == tc::EW) {
        // ===== MMA issuer (one elected lane).  The column blocks of the accumulator advance INDEPENDENTLY: a block's next
        // group is issued as soon as its ray tile is there and its columns of the buffer have been read =====
        if (lane == 0) {
            const unsigned total = n_it * (unsigned)tiles;
            unsigned gi[tc::NBLK];                              // groups issued per block
#pragma unroll
            for (int c = 0; c < tc::NBLK; ++c) gi[c] = 0;
            unsigned ready_tiles = 0, freed_tiles = 0;
            const uint32_t b_base = tc::smem_u32(S.B);
            for (unsigned idle = 0;;) {
                bool left = false, progressed = false;
#pragma unroll
                for (int c = 0; c < tc::NBLK; ++c) {
                    const unsigned gq = gi[c];
                    if (gq >= total) continue;
                    left = true;
                    const unsigned it = gq / (unsigned)tiles, jt = gq - it * (unsigned)tiles, s = it % slots, b = gq & 1u;
                    if (it >= ready_tiles) {                    // tiles become ready in order
                        if (!tc::mbar_try_wait(&S.a_ready[s], (it / slots) & 1u)) continue;
                        ready_tiles = it + 1;
                    }
                    if (!tc::mbar_try_wait(&S.d_empty[b * tc::NBLK + c], ((gq >> 1) & 1u) ^ 1u)) continue;
                    tc::fence_after();
                    const uint32_t a_addr = tc::smem_u32(S.A(s));
                    const uint32_t b_addr = b_base + jt * tc::B_TILE_BYTES + (uint32_t)c * (tc::BLOCK_N / 8) * 128;
#pragma unroll
                    for (int kk = 0; kk < tc::KTOT / 8; ++kk)
                        tc::mma_tf32(tmem + b * tc::TILE_N + (uint32_t)c * tc::BLOCK_N, tc::make_desc(a_addr + kk * 2 * tc::TILE_M * 16, tc::TILE_M * 16, 128),
                                     tc::make_desc(b_addr + kk * 2 * tc::TILE_N * 16, tc::TILE_N * 16, 128), kk > 0);
                    tc::mma_commit(&S.d_full[b * tc::NBLK + c]);
                    gi[c] = gq + 1;
                    progressed = true;
                }
                // a ray tile's buffer is free once EVERY block has issued all its groups of that tile
                unsigned mn = gi[0];
#pragma unroll
                for (int c = 1; c < tc::NBLK; ++c) mn = min(mn, gi[c]);
                for (const unsigned done = mn / (unsigned)tiles; freed_tiles < done; ++freed_tiles) tc::mma_commit(&S.a_free[freed_tiles % slots]);
                if (!left) break;
                if (progressed) idle = 0;
                else if (++idle > 0x20000000u) __trap();        // a protocol error must not hang the device
            }
            // the last commit's arrival is asynchronous: it must have landed in this CTA's shared memory before the CTA may exit
            tc::mbar_wait(&S.a_free[(n_it - 1) % slots], ((n_it - 1) / slots) & 1u);
        }
        __syncwarp();
    } else {
        // ===== epilogue warps: warp w reads TMEM lanes 32 (w % 4).., columns 64 (w / 4).. of every accumulator =====
        const unsigned rl = (warp & 3u) * 32u + lane;          // this thread's ray within the tile = its TMEM lane
        const unsigned cb = warp >> 2;                          // this warp's 64 columns of a buffer
        const unsigned blk = warp / tc::BLOCK_WARPS;            // the independently advancing column block they belong to
        const uint32_t t_lane = ((warp & 3u) * 32u) << 16;
        uint32_t* cand = S.cand + warp * tc::CAND_CAP;
        unsigned* cand_n = S.cand_n + warp;
        TcEmit E{0u, 0u, 0u, false, 0u};
        unsigned g = 0;
        for (unsigned it = 0; it < n_it; ++it) {
            const unsigned s = it % slots, a_ph = (it / slots) & 1u, tile = first + it;
            for (int j = 0; j < tiles; ++j, ++g) {
                const unsigned b = g & 1u;
                TC_T(t0);
                tc::mbar_wait(&S.d_full[b * tc::NBLK + blk], (g >> 1) & 1u);
                TC_ACC(0, t0);
                tc::fence_after();
                const uint32_t taddr = tmem + t_lane + b * tc::TILE_N + cb * 64u;
                unsigned m0, m1;
                TC_T(t1);
                {
                    uint32_t v0[32], v1[32];
                    RT_TMEM_LD32(taddr, v0);
                    RT_TMEM_LD32(taddr + 32u, v1);
                    tc::tmem_wait_ld();
                    tc::fence_before();                         // the 64 columns are in registers: hand them back
                    __syncwarp();
                    if (lane == 0) tc::mbar_arrive(&S.d_empty[b * tc::NBLK + blk]);
                    unsigned w0 = 0u, w1 = 0u;
#pragma unroll
                    for (int q = 0; q < 32; ++q) { w0 = __funnelshift_l(v0[q], w0, 1); w1 = __funnelshift_l(v1[q], w1, 1); }
                    const bool live_ray = tile * tc::TILE_M + rl < n;   // (a dead ray's discriminants are all -1e30; never let it index anything)
                    m0 = live_ray ? ~w0 : 0u; m1 = live_ray ? ~w1 : 0u;   // candidates: clear sign bits; column q of a word is bit 31 - q
                }
                TC_ACC(1, t1);
                TC_T(t2);
                const unsigned row0 = (unsigned)j * tc::TILE_N + cb * 64u;
#ifdef RT_TC_CHECK
                {   // the accumulator's sign bits against the same products summed in double from the operands in shared memory
                    const unsigned char* Ab = reinterpret_cast<const unsigned char*>(S.A(s));
                    const unsigned char* Bb = reinterpret_cast<const unsigned char*>(S.B) + (size_t)j * tc::B_TILE_BYTES;
                    for (int q = 0; q < 64; ++q) {
                        double acc = 0.0, mag = 0.0;
                        for (int k = 0; k < tc::KTOT; ++k) {
                            const double x = (double)*reinterpret_cast<const float*>(Ab + tc::canon_off(tc::TILE_M, (int)rl, k)) *
                                             (double)*reinterpret_cast<const float*>(Bb + tc::canon_off(tc::TILE_N, (int)(cb * 64u) + q, k));
                            acc += x; mag += fabs(x);
                        }
                        const unsigned culled = ((q < 32 ? ~m0 : ~m1) >> (31 - (q & 31))) & 1u;   // sign bit as collected
                        if (acc > 1e-4 * mag && culled && mag < 1e20)
                            printf("TMEM mismatch: tile %u ray %u col %u (row %u) double %g (mag %g) but sign bit set; block %u warp %u buffer %u g %u\n", tile, rl, (unsigned)q, row0 + q,
                                   acc, mag, blockIdx.x, warp, b, g);
                        if (acc < -1e-4 * mag && !culled)
                            printf("TMEM mismatch: tile %u ray %u col %u (row %u) double %g (mag %g) but sign bit clear; block %u warp %u buffer %u g %u\n", tile, rl, (unsigned)q, row0 + q,
                                   acc, mag, blockIdx.x, warp, b, g);
                    }
                }
#endif
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    unsigned mm = h ? m1 : m0;
                    while (mm != 0u) {                          // lanes with candidates only (divergent; a shared-memory atomic hands out slots)
                        const int bit = 31 - __clz((int)mm);
                        mm &= ~(1u << bit);
                        const unsigned pos = atomicAdd(cand_n, 1u);
                        if (pos < (unsigned)tc::CAND_CAP) cand[pos] = (rl << 20) | (row0 + (unsigned)h * 32u + (unsigned)(31 - bit));   // (a full list: see below)
                    }
                }
                TC_ACC(2, t2);
            }
            TC_T(t3);
            __syncwarp();
            const unsigned raw = *cand_n;                       // every push counted, also those that found the list full
            const bool overflowed = raw > (unsigned)tc::CAND_CAP;   // then: drop the list, redo this warp's share of the tile in FP32
            const unsigned ncand = overflowed ? 0u : raw;
            if (overflowed) {
                tc::mbar_wait(&S.a_ready[s], a_ph);
                tc_redo_fp32(W, S, (int)s, tile, n, n_g, n_p, tiles, cb, rl);
                __syncwarp();
            }
#ifdef RT_TC_CHECK
            if (lane == 0 && ncand > 48u && n < 300u)
                printf("big candidate list: block %u warp %u tile %u it %u ncand %u raw %u first %x %x %x %x last %x\n", blockIdx.x, warp, tile, it, ncand, raw, cand[0], cand[1], cand[2], cand[3], cand[ncand - 1]);
#endif
            if (ncand) {
                tc::mbar_wait(&S.a_ready[s], a_ph);             // (long complete) the producers' writes of ray[s], acquired directly
                tc_drain(W, S, (int)s, tile, n_g, n_p, cand, ncand, E, lane);
            }
            __syncwarp();
            if (lane == 0) {
                *cand_n = 0u;
                tc::mbar_arrive(&S.ray_free[s]);
            }
            __syncwarp();
            TC_ACC(3, t3);
        }
        tc_pad(W, E, E.pos, E.end, lane);
        if (E.ahead) {                 // the reservation requested ahead and never used
            const unsigned b = __shfl_sync(0xffffffffu, E.next, 0);
            tc_pad(W, E, min(b, W.pair_cap), min(b + (unsigned)tc::PAIR_CHUNK, W.pair_cap), lane);
            if (lane == 0 && E.pads) atomicAdd(&W.st->pad, E.pads);
        }
    }
#ifdef RT_TC_TIMING
    if (blockIdx.x == 0 && lane == 0 && n_it > 8)
        printf("tc warp %2u (%s) tiles %u total %lld : %lld %lld %lld %lld cycles per tile\n", warp, warp < tc::EW ? "epi: d_full wait, ld+shf, cand, drain" : (warp == tc::EW ? "mma: a_ready wait, d_empty wait, issue" : "prod: a_free wait, ray_free wait, produce"),
               n_it, (clock64() - t_begin) / n_it, tacc[0] / n_it, tacc[1] / n_it, tacc[2] / n_it, tacc[3] / n_it);
#endif
    tc::fence_before();
    __syncthreads();
    if (warp == tc::EW) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
}

// ------------------------------------------------------------------------------------------
// rt_cull_check with cull_tc = 1: the PRODUCTION kernel above runs over a queue that holds the caller's rays, then every
// (ray, listed leaf) the exact FP64 test accepts must be among the emitted pairs.
// ------------------------------------------------------------------------------------------
__global__ void tc_check_fill(const __grid_constant__ WaveParams W, int n, const float* origins, const float* dirs, const float* times) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) {
        WaveState* st = W.st;
        st->cnt[0][0] = (unsigned)n; st->cnt[0][1] = 0; st->cnt[1][0] = 0; st->cnt[1][1] = 0;
        st->gen_base[0] = 0; st->gen_base[1] = 0;
        st->batch = 0; st->npairs = 0; st->exhausted = 1; st->done = 0; st->mode = MODE_RUN; st->pad = 0;
    }
    if (i >= n) return;
    float4* q = W.queue[0] + 3 * (size_t)i;
    q[0] = make_float4(origins[3 * i], origins[3 * i + 1], origins[3 * i + 2], times ? times[i] : 0.f);
    q[1] = make_float4(dirs[3 * i], dirs[3 * i + 1], dirs[3 * i + 2], 0.f);
    q[2] = make_float4(0.f, 0.f, 0.f, 0.f);
}
__global__ void tc_check_mark(const __grid_constant__ WaveParams W, unsigned* mask, int words) {
    const unsigned npairs = min(W.st->npairs, W.pair_cap);
#ifdef RT_TC_CHECK
    if (blockIdx.x == 0 && threadIdx.x == 0 && W.st->cnt[0][0] < 300u) {
        // the harness filled the pair buffer with 0xDD bytes: a slot still holding them was never written
        for (unsigned c0 = 0; c0 < npairs; c0 += 64) {
            unsigned never = 0, real = 0, tag0 = 0xffffffffu, tags = 0;
            for (unsigned i = c0; i < min(c0 + 64u, npairs); ++i) {
                const uint2 pr = W.pairs[i];
                if (pr.x == 0xddddddddu) ++never;
                else if (pr.x == PAIR_NULL) { if (pr.y != tag0) { ++tags; tag0 = pr.y; } }
                else ++real;
            }
            if (never || tags > 1 || real)
                printf("chunk %u: never written %u, real %u, pad-tag changes %u (last tag block %u warp %u)  first entries (%x %x) (%x %x) (%x %x) ... (%x %x)\n", c0, never, real, tags,
                       tag0 >> 8, tag0 & 255u, W.pairs[c0].x, W.pairs[c0].y, W.pairs[c0 + 1].x, W.pairs[c0 + 1].y, W.pairs[c0 + 2].x, W.pairs[c0 + 2].y, W.pairs[c0 + 63].x, W.pairs[c0 + 63].y);
        }
        printf("npairs %u pad counter %u\n", W.st->npairs, W.st->pad);
    }
#endif
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < npairs; i += gridDim.x * blockDim.x) {
        const uint2 pr = W.pairs[i];
        if (pr.x != PAIR_NULL && pr.x < (unsigned)W.capacity) atomicOr(&mask[(size_t)pr.x * words + (pr.y >> 5)], 1u << (pr.y & 31u));
    }
}
__global__ void __launch_bounds__(128) tc_check_compare(const __grid_constant__ WaveParams W, int n, double tmin, double tmax, const unsigned* mask,
                                                        int words, unsigned long long* out) {
    const DevScene& sc = W.base.sc;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long lost = 0, surv = 0, cand = 0;
    if (idx < n) {
        const float4 a = W.queue[0][3 * (size_t)idx], b = W.queue[0][3 * (size_t)idx + 1];
        const bool overflow = W.best_key[idx] == BEST_KEY_OVERFLOW;      // its pairs did not fit: re-intersected exactly downstream
        for (int k = 0; k < sc.n_list; ++k) {
            const bool kept = overflow || ((mask[(size_t)idx * words + (k >> 5)] >> (k & 31)) & 1u);
            const double t = sc.generic ? refine_leaf<true>(&W.base.sc, k, a.x, a.y, a.z, b.x, b.y, b.z, a.w, tmin, tmax, false, make_uint2(0u, 0u), 0u, 0u, 0u)
                                        : refine_leaf<false>(&W.base.sc, k, a.x, a.y, a.z, b.x, b.y, b.z, a.w, tmin, tmax, false, make_uint2(0u, 0u), 0u, 0u, 0u);
            surv += kept ? 1u : 0u;
            if (t < CUDART_INF) {
                cand++;
                lost += kept ? 0u : 1u;
#ifdef RT_TC_CHECK
                if (!kept) printf("lost pair: ray %d leaf %d t %.9g  o (%.9g %.9g %.9g) d (%.9g %.9g %.9g)\n", idx, k, t, a.x, a.y, a.z, b.x, b.y, b.z);
#endif
            }
        }
    }
    if (lost) atomicAdd(&out[0], lost);
    if (surv) atomicAdd(&out[1], surv);
    if (cand) atomicAdd(&out[2], cand);
}
