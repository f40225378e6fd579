/*
 * raytrace_b200.h — C ABI of libraytrace_b200.so
 *
 * The drop-in boundary for ONE hot path of gonewest818/raytrace-clj: the per-pixel
 * path-tracing loop.  The reference has no FFI of its own; the seam is the render
 * block of `-main` (reference src/raytrace_clj/core.clj:99-108): input
 * (nx ny nr camera world), output every pixel's [ir ig ib] written at
 * (i, ny-1-j).  Everything the reference computes inside that block — `pixel`
 * (core.clj:43-57), `color` (core.clj:17-41), `get-ray` (camera.clj:8-16,35-48),
 * `hit?` on Sphere / UVSphere / MovingSphere and the brute-force closest-hit
 * reduce (hitable.clj:15-26,141-259), `scatter`/`emitted` of Lambertian / Metal /
 * Dielectric / DiffuseLight (shader.clj:6-119), `sample` of Constant / UVGradient
 * / Checkerboard (texture.clj:14-50) and the vec3 helpers (util.clj:5-52) — runs
 * on the GPU behind these entry points.
 *
 * Conventions
 *   - plain pointers and sizes only; the caller owns every host buffer, the
 *     library copies during the call and keeps no host pointer after return;
 *   - every function returns RT_OK (0) or a negative rt_status; the message of
 *     the last failure on a context is `rt_last_error(ctx)`;
 *   - one rt_ctx may be used by one thread at a time (calls are serialised by a
 *     mutex inside the context);
 *   - there is NO CPU fallback: without a usable CUDA device rt_create fails.
 *
 * The JVM-side binding (JNA) a maintainer would add to the reference is shown in
 * INTEGRATION.md and shipped as source under clojure/.
 */
#ifndef RAYTRACE_B200_H
#define RAYTRACE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_ABI_VERSION 2   /* 2: + rt_set_scene_ex / rt_scene_ext, rt_trace_paths, rt_set_accel, rt_set_option, rt_sample_device (additive) */
                           /* (rt_host_alloc / rt_host_free joined version 2 later: additive, optional — an older library simply lacks the symbols) */

typedef struct rt_ctx rt_ctx;

typedef enum rt_status {
    RT_OK = 0,
    RT_ERR_ARG = -1,          /* bad argument (null pointer, negative size, bad id …)   */
    RT_ERR_UNSUPPORTED = -2,  /* object / material / texture type outside the hot path  */
    RT_ERR_CUDA = -3,         /* CUDA runtime error; rt_last_error has the CUDA string  */
    RT_ERR_STATE = -4,        /* call order: render before set_scene / set_camera       */
    RT_ERR_NODEVICE = -5,     /* no usable CUDA device (there is no CPU fallback)       */
    RT_ERR_NCCL = -6          /* NCCL not loadable / a collective failed (multi-device reduce) */
} rt_status;

/* sphere_flags bits */
#define RT_SPHERE_UV      1u  /* UVSphere (hitable.clj:141-172): uv from get-sphere-uv (hitable.clj:128-139) */
#define RT_SPHERE_MOVING  2u  /* MovingSphere (hitable.clj:224-259): centre lerped by ray time                */

/* material types (shader.clj) */
#define RT_MAT_LAMBERTIAN    0  /* shader.clj:29-36   tex = albedo                    */
#define RT_MAT_METAL         1  /* shader.clj:46-59   tex = albedo, param = fuzz      */
#define RT_MAT_DIELECTRIC    2  /* shader.clj:76-104  param = ri                      */
#define RT_MAT_DIFFUSE_LIGHT 3  /* shader.clj:114-119 tex = emission                  */

#define RT_MAT_ISOTROPIC     4  /* shader.clj:129-138 tex = albedo; scattered ray time = hit t (as in the reference); rt_set_scene_ex only */

/* texture types (texture.clj) */
#define RT_TEX_CONSTANT      0  /* texture.clj:14-16  params[0..2] = colour                                  */
#define RT_TEX_UV_GRADIENT   1  /* texture.clj:26-34  params = co[3] cu[3] cv[3] cuv[3]                       */
#define RT_TEX_CHECKERBOARD  2  /* texture.clj:44-50  params[0] = scale, children = {tex0, tex1}              */
/* the following need rt_set_scene_ex (Perlin tables / images travel in rt_scene_ext) */
#define RT_TEX_PERLIN_NOISE  3  /* texture.clj:60-64  params[0] = scale                                       */
#define RT_TEX_PERLIN_TURB   4  /* texture.clj:74-78  params[0] = scale, params[1] = depth                    */
#define RT_TEX_MARBLE        5  /* texture.clj:88-93  params[0] = scale, params[1] = depth                    */
#define RT_TEX_FLIP_U        6  /* texture.clj:103-106 children[0] = tex                                      */
#define RT_TEX_FLIP_V        7  /* texture.clj:113-116 children[0] = tex                                      */
#define RT_TEX_IMAGE_MAP     8  /* texture.clj:126-133 params[0] = image index (indices clamped to the image) */

/* primitive types (hitable.clj), rt_scene_ext.prim_type */
#define RT_PRIM_SPHERE    0  /* Sphere / UVSphere / MovingSphere: center0_r, center1, t0t1, sphere_flags as in rt_scene_desc */
#define RT_PRIM_RECT_XY   1  /* hitable.clj:272-297  prim_params = x0 y0 x1 y1 k   (inclusive t range, unlike spheres)      */
#define RT_PRIM_RECT_XZ   2  /* hitable.clj:303-328  prim_params = x0 z0 x1 z1 k                                            */
#define RT_PRIM_RECT_YZ   3  /* hitable.clj:334-359  prim_params = y0 z0 y1 z1 k                                            */
#define RT_PRIM_TRIANGLE  4  /* hitable.clj:548-581  prim_params = v0 v1 v2 (9 floats); single-sided, un-normalised normal  */
#define RT_PRIM_MEDIUM    5  /* hitable.clj:516-543  ConstantMedium: prim_params[0] = density, prim_aux = {first boundary
                                primitive, count} (a sphere: 1; a Box: its 6 rectangles); material = RT_MAT_ISOTROPIC          */

/* wrapper ops folded into a leaf's transform chain, outermost first (rt_scene_ext.xform_ops) */
#define RT_XOP_NONE       0
#define RT_XOP_TRANSLATE  1  /* hitable.clj:391-405  params = offset x y z   */
#define RT_XOP_ROTATE_Y   2  /* hitable.clj:410-486  params = sin(theta), cos(theta) */
#define RT_XOP_FLIP       3  /* hitable.clj:375-386  FlipNormals             */
#define RT_XFORM_MAX_OPS  4

/* which leaf wins an EXACT tie in t (coincident geometry only) */
#define RT_TIE_HITLIST    0  /* the world is a Hitlist (hitable.clj:15-26): the first sphere in caller order, but a later
                                rectangle / triangle (inclusive range test) replaces an equal earlier hit                    */
#define RT_TIE_BVH        1  /* the world is a bvh-node tree (hitable.clj:97-106, right child wins): the LAST leaf in flatten order */

/* closest-hit search (rt_set_accel) */
#define RT_ACCEL_BRUTE_FORCE 0  /* FP32 cull over ALL listed primitives per ray: the roofline path (default)                 */
#define RT_ACCEL_BVH         1  /* flattened GPU BVH feeding the same FP64 refine: the role of hitable.clj:97-123             */

/* how a path ended (rt_trace_paths out_term) */
#define RT_TERM_LIGHT   1
#define RT_TERM_ABSORB  2
#define RT_TERM_DEPTH   3
#define RT_TERM_MISS    4

/* camera types (camera.clj) */
#define RT_CAM_PINHOLE    0     /* camera.clj:8-16   uses origin, lleft, horiz, vert; ray time 0, no RNG draws */
#define RT_CAM_THIN_LENS  1     /* camera.clj:35-48  all 24 floats                                             */

/* render variants */
#define RT_VARIANT_MEGAKERNEL 0 /* persistent megakernel with per-lane path regeneration */
#define RT_VARIANT_WAVEFRONT  1 /* persistent wavefront: generate / intersect / shade / compact queues */

/*
 * Scene = the flattened leaves of the reference's `world` (hitable.clj:97-123 bvh-node
 * tree walked left to right, de-duplicated), as structure-of-arrays host buffers.
 * Replaces: the Hitable / Shader / Texture record graph reachable from `world`
 * (core.clj:90).  float32 on the wire; the reference holds doubles.
 */
typedef struct rt_scene_desc {
    int32_t n_spheres;
    const float* center0_r;        /* 4*n: cx cy cz radius            (Sphere/UVSphere centre, MovingSphere centre0) */
    const float* center1;          /* 4*n: c1x c1y c1z pad, or NULL   (MovingSphere centre1; ignored if not moving)  */
    const float* t0t1;             /* 2*n: t0 t1, or NULL             (MovingSphere t0 t1)                           */
    const uint32_t* sphere_flags;  /* n: RT_SPHERE_* bits                                                            */
    const int32_t* material_id;    /* n: index into the material table                                               */
    int32_t n_materials;
    const int32_t* mat_type;       /* m: RT_MAT_*                                                                    */
    const float* mat_param;        /* m: fuzz (metal) | ri (dielectric) | unused                                     */
    const int32_t* mat_tex;        /* m: texture id (albedo / emission) or -1                                        */
    int32_t n_textures;
    const int32_t* tex_type;       /* t: RT_TEX_*                                                                    */
    const float* tex_params;       /* 12*t                                                                           */
    const int32_t* tex_children;   /* 2*t: child texture ids (checkerboard) or -1                                    */
} rt_scene_desc;

/*
 * Everything beyond spheres and the three basic textures (ABI 2, additive: rt_scene_desc is unchanged).
 * Every per-primitive array of rt_scene_desc AND of this struct then holds n_spheres WORLD primitives (flatten
 * order) followed by n_boundary BOUNDARY primitives (the boundaries of media; never hit directly).
 * Replaces: RectXY/XZ/YZ, FlipNormals, Translate, RotateY, Box, ConstantMedium, Triangle (hitable.clj:269-581),
 * Isotropic (shader.clj:129-143), PerlinNoise/Turbulence/Marble/FlipTexture/ImageMap (texture.clj:60-138) and
 * the Perlin tables perlin.clj:6-17 (marshalled: the reference draws them from the unseeded RNG at load time).
 */
typedef struct rt_scene_ext {
    int32_t struct_bytes;          /* sizeof(rt_scene_ext) as the caller knows it                                   */
    int32_t n_boundary;            /* boundary primitives after the n_spheres world primitives                       */
    const int32_t* prim_type;      /* n_spheres + n_boundary: RT_PRIM_*; NULL => all spheres                         */
    const float* prim_params;      /* 12 * (n_spheres + n_boundary)                                                  */
    const int32_t* prim_aux;       /* 2 * (n_spheres + n_boundary): medium = {first boundary primitive, count}       */
    const int32_t* prim_xform;     /* n_spheres + n_boundary: index into the transform table or -1                   */
    int32_t n_xforms;
    const int32_t* xform_ops;      /* RT_XFORM_MAX_OPS * n_xforms: RT_XOP_*, outermost wrapper first, 0-terminated   */
    const float* xform_params;     /* 4 floats per op                                                                */
    int32_t tie_rule;              /* RT_TIE_*                                                                       */
    const float* perlin_vectors;   /* 256 * 3 (perlin.clj:6-8) or NULL                                               */
    const int32_t* perlin_perm;    /* 3 * 256: perm-x, perm-y, perm-z (perlin.clj:10-17) or NULL                      */
    int32_t n_images;
    const int32_t* image_wh;       /* 2 * n_images: width, height                                                    */
    const int64_t* image_offset;   /* n_images: byte offset of image i in image_rgb                                  */
    const uint8_t* image_rgb;      /* RGB bytes, rows top to bottom (imagez get-pixel x y)                           */
} rt_scene_ext;

/* one logged ray of rt_trace_paths */
typedef struct rt_path_bounce {
    float o[3];
    float time;
    float d[3];
    int32_t hit_id;                /* caller's primitive index, -1 = miss, -2 = the path had ended before this bounce */
    double t;
} rt_path_bounce;

/*
 * Camera record (camera.clj:35 ThinLensCamera / camera.clj:8 PinholeCamera):
 * cam[0..20] = origin lleft horiz vert u v w (3 floats each), cam[21] = aperture,
 * cam[22] = t0, cam[23] = t1.
 */

/* counters filled by rt_get_counters (the reference's metrics.clj:7-9 counters, on device) */
enum {
    RT_CTR_RAYS = 0,         /* hit?(world) calls  == `total-rays` (core.clj:24)                  */
    RT_CTR_SPHERE_TESTS,     /* ray-sphere discriminant evaluations == rays * n_spheres           */
    RT_CTR_SAMPLES,          /* top-level `color` calls (core.clj:51)                             */
    RT_CTR_TERM_LIGHT,       /* paths ended on a non-scattering material (DiffuseLight)           */
    RT_CTR_TERM_ABSORB,      /* paths ended by Metal.scatter returning nil (shader.clj:54)        */
    RT_CTR_TERM_DEPTH,       /* paths ended by the depth cutoff (core.clj:26)                     */
    RT_CTR_TERM_MISS,        /* paths ended by a miss (core.clj:40-41)                            */
    RT_CTR_KERNEL_NS,        /* device time of the last render's kernels, ns (CUDA events)        */
    RT_CTR_CANDIDATES,       /* (ray, sphere) pairs that passed the FP32 cull and were refined    */
    RT_CTR_KERNEL_LAUNCHES,  /* CUDA kernels launched by this context (render + resolve + diagnostics) */
    RT_CTR_CULL_NS,          /* with rt_set_profile(ctx, 1): device time per wavefront stage, ns  */
    RT_CTR_REFINE_NS,
    RT_CTR_TIEBREAK_NS,
    RT_CTR_SHADE_NS,
    RT_CTR_DIRECT_TESTS,     /* exact (FP64) tests of the few enclosing spheres that bypass the FP32 cull (counted apart
                                from the culled tests; RT_CTR_SPHERE_TESTS = rays * n still counts every pair once)   */
    RT_CTR_BVH_NODE_TESTS,   /* RT_ACCEL_BVH: box tests (the reference's `aabb.intersection.total`, metrics.clj:9)     */
    RT_CTR_REDUCE_NS,        /* multi-device rt_render: device time of the cross-device reduce, ns                     */
    RT_CTR_COUNT = 24
};

/* ---- lifecycle ------------------------------------------------------------------------ */

/* Create a context on `n_devices` CUDA devices (ids in device_ids; NULL => device 0).
 * n_devices > 1 renders sample slices on every device from this one process and combines
 * the per-device float sums on device_ids[0] over NVLink peer access.                        */
int rt_create(rt_ctx** out, const int* device_ids, int n_devices);
void rt_destroy(rt_ctx* ctx);
const char* rt_last_error(const rt_ctx* ctx);   /* ctx may be NULL: last rt_create failure */
int rt_abi_version(void);

/* ---- scene / camera (replace the record graph built at core.clj:82-90) ---------------- */
int rt_set_scene(rt_ctx* ctx, const rt_scene_desc* scene);
/* the same with the extension record (ext may be NULL = rt_set_scene) */
int rt_set_scene_ex(rt_ctx* ctx, const rt_scene_desc* scene, const rt_scene_ext* ext);
/* rt_set_scene for a scene whose PER-PRIMITIVE arrays live in device memory on the context's first device:
 * center0_r, center1, t0t1, sphere_flags, material_id are DEVICE pointers (center1 / t0t1 / sphere_flags may be NULL as
 * in rt_set_scene); the material and texture tables stay HOST pointers.  Spheres / UVSpheres / MovingSpheres with the
 * four rt_set_scene materials and three textures only (everything rt_set_scene accepts; nothing of rt_scene_ext).
 * The library orders its reads after the work already enqueued on `stream` (a cudaStream_t, NULL = legacy default);
 * it returns once the scene is built, so the caller may overwrite or free the arrays afterwards.
 * Same validation, status codes and messages as rt_set_scene; a rejected scene leaves the previous one in place.
 * The scene then behaves exactly as if rt_set_scene had been given the same values: the GPU builds the same blob bytes
 * (the host's marshalling restated kernel by kernel), so a caller whose spheres are already on the GPU (a simulation, a
 * generated scene) skips the copy to the host, the single-threaded marshalling and the upload.  A per-primitive pointer
 * that is not device or managed memory of device_ids[0] -> RT_ERR_ARG.  Added within ABI version 2, like rt_get_bvh. */
int rt_set_scene_device(rt_ctx* ctx, const rt_scene_desc* scene, void* stream);
/* The scene blob device `device_index` holds (diagnostic): out may be NULL to query *bytes; otherwise cap >= *bytes.
 * Added within ABI version 2.                                                                                       */
int rt_get_scene_blob(rt_ctx* ctx, int device_index, void* out, size_t cap, size_t* bytes);
/* closest-hit search used by the renders that follow: RT_ACCEL_BRUTE_FORCE (default) or RT_ACCEL_BVH */
int rt_set_accel(rt_ctx* ctx, int accel);
/* Per-context tuning knob; the RT_* environment variables only give the defaults at rt_create.  Names:
 * "wave_lanes", "wave_capacity", "cull_claims", "cull_ctas_per_sm", "light_block", "tail_entries", "tile_records",
 * "direct_spheres", "common_origin", "reduce" (0 peer loads in the resolve kernel, 1 ncclReduce), "rows" (multi-device
 * partition: 0 sample slices, 1 interleaved rows), "cull_tc" (1 = the brute-force cull runs on the tensor cores when the
 * list has 160 leaves or more, all spheres (default), 0 = FP32 pipe only, 2 = FP32 for a lane's first all-camera-ray iteration, 3 = tensor
 * cores whatever the list length),
 * "tc_tiles_per_cta", "tc_ctas", "wave_depth", "tail_rays", "tail_solo" (a tail slice of this many paths or fewer runs one warp per
 * path, default 24; 0 = staged to the end), "tail_lpp" (lanes per such path: 8 | 16 | 32), "tail_block", "cull_shape",
 * "tail_ctas_per_sm", "mega_regcap", "bvh_build" (where RT_ACCEL_BVH's tree is built: 1 = on the device from 1000 listed leaves
 * up, on the host below (default), 0 = host always, 2 = device always; a device tree deeper than the traversal's 48-entry
 * stack is replaced by the host build before any ray sees it).
 * Unknown name -> RT_ERR_ARG.                                                                                     */
int rt_set_option(rt_ctx* ctx, const char* name, int64_t value);
int rt_set_camera(rt_ctx* ctx, int cam_type, const float cam[24]);

/* ---- the hot path (replaces core.clj:99-108) ------------------------------------------ */

/* Limits (checked, RT_ERR_ARG): nx * ny <= (2^31 - 1) / 3 pixels; nsamples (and sample_begin + sample_count) < 2^24;
 * the wavefront variant packs the remaining depth in 8 bits: max_depth <= 255 (the megakernel takes any depth >= 0).
 *
 * Render nsamples per pixel, depth cutoff max_depth (reference: 50, core.clj:20,45).
 * out_linear_rgb: nx*ny*3 float, per-pixel SUM over samples / nsamples (before gamma),
 *                 pixel (i, j) at ((j*nx)+i)*3, j = 0 is the BOTTOM row (reference's j); may be NULL.
 * out_rgb8:       nx*ny*3 bytes after sqrt, *255.99, min, truncate (core.clj:52-57), row 0 = TOP
 *                 (reference writes row ny-1-j, core.clj:105); may be NULL.                      */
int rt_render(rt_ctx* ctx, int nx, int ny, int nsamples, int max_depth, uint64_t seed,
              int variant, float* out_linear_rgb, uint8_t* out_rgb8);

/* Page-locked host memory for rt_render's outputs (what the reference holds in its BufferedImage, core.clj:100-108).
 * rt_render recognises a page-locked destination — from here, or any buffer the caller registered with the CUDA runtime —
 * and has the device write the result into it directly; into ordinary pageable memory the result goes through the
 * context's own page-locked staging buffer plus one host copy.  A JNA / JNI caller wraps the pointer as a direct
 * ByteBuffer.  ctx may be NULL (the memory is usable with every context of the process).        */
int rt_host_alloc(rt_ctx* ctx, size_t bytes, void** out);
int rt_host_free(rt_ctx* ctx, void* p);

/* The RT_ACCEL_BVH tree as device `device_index` of the context holds it (built first if the scene or the movers' time
 * window changed since the last build, whatever the accelerator): 16 floats per node (left child's box lo.xyz hi.xyz,
 * right child's box lo.xyz hi.xyz, then left, right, 0, 0 as int32; a leaf child k in cull order is stored as ~k; the root is
 * node 0).  out_nodes may be NULL; otherwise cap_nodes must be at least the node count.  info = {node count, depth of the
 * deepest leaf (root = 0), builder (0 host, 1 device), device build time in ns from CUDA events (0 for the host build)}.
 * Added within ABI version 2, like rt_host_alloc / rt_host_free.                                                        */
int rt_get_bvh(rt_ctx* ctx, int device_index, float* out_nodes, int64_t cap_nodes, int64_t info[4]);

/* Same render, device-resident: accumulate samples [sample_begin, sample_begin+sample_count)
 * of every pixel whose row j satisfies j % row_stride == row_offset into d_sum (DEVICE pointer on
 * the context's first device, nx*ny*3 float, += semantics; caller zeroes it).  This is the
 * per-GPU leg of a sharded render: the caller reduces d_sum across ranks (NCCL) and then calls
 * rt_resolve_device.  Launches on `stream` (a cudaStream_t cast to void*, NULL = default).
 * Returns after the kernels are enqueued if `sync` is 0.                                       */
int rt_render_accumulate_device(rt_ctx* ctx, int nx, int ny, int sample_begin, int sample_count,
                                int row_offset, int row_stride, int max_depth, uint64_t seed,
                                int variant, float* d_sum, void* stream, int sync);

/* core.clj:52-57 on the device: out = int(min(255.99, 255.99*sqrt(sum/nsamples_total))), y-flipped.
 * d_rgb8 is a DEVICE pointer (nx*ny*3 bytes).                                                   */
int rt_resolve_device(rt_ctx* ctx, int nx, int ny, int nsamples_total, const float* d_sum,
                      uint8_t* d_rgb8, void* stream, int sync);

/* ---- diagnostics used by the parity tests ---------------------------------------------- */

/* Closest hit of n caller-given rays against the scene = Hitlist.hit? (hitable.clj:15-26)
 * over the flattened leaves: out_t[i] (double, +inf on a miss), out_id[i] = sphere index or -1.  */
int rt_trace_primary(rt_ctx* ctx, int n, const float* origins /*3n*/, const float* dirs /*3n*/,
                     const float* times /*n or NULL*/, double tmin, double tmax,
                     double* out_t, int32_t* out_id);

/* The production render code (either variant: same queues / cull / refine / shade kernels) run for n caller-chosen
 * (pixel, sample) pairs of an nx x ny frame instead of the whole frame: pixel[q] = j * nx + i (j = 0 bottom row),
 * sample[q] = the sample index keyed into the Philox counters.  Per path: out_radiance (3n, what `color` returns,
 * core.clj:17-41), out_nrays (hit?(world) calls), out_term (RT_TERM_*); out_log (n * log_bounces records or NULL)
 * receives the first log_bounces rays of every path with the hit the renderer resolved for them.               */
int rt_trace_paths(rt_ctx* ctx, int nx, int ny, int n, const int32_t* pixel, const int32_t* sample, int max_depth,
                   uint64_t seed, int variant, float* out_radiance, int32_t* out_nrays, int32_t* out_term,
                   int log_bounces, rt_path_bounce* out_log);

/* n points of the device's rand-in-unit-sphere (kind 0: 3n floats) or rand-in-unit-disk (kind 1: 2n floats) —
 * util.clj:32-52 in closed form — drawn from the Philox counters (pixel = index, sample 0, bounce 1 | 0).       */
int rt_sample_device(rt_ctx* ctx, int kind, int n, uint64_t seed, float* out);

/* The contract of the FP32 cull (the brute-force loop over the sphere list), checked pair by pair on the
 * device: out[0] = (ray, listed sphere) pairs whose exact FP64 test (hitable.clj:185-206) accepts a root in
 * (tmin, tmax) but whose FP32 cull key says "cannot hit" — must be 0; out[1] = pairs the cull lets through;
 * out[2] = pairs the exact test accepts.  tmin >= 0 (as for rt_trace_primary).                            */
int rt_cull_check(rt_ctx* ctx, int n, const float* origins /*3n*/, const float* dirs /*3n*/,
                  const float* times /*n or NULL*/, double tmin, double tmax, uint64_t out[3]);

/* Camera rays exactly as the render kernels generate them for (pixel i, j, sample s):
 * out_origin/out_dir 3n floats, out_time n floats; ij is 2n int32 (i, j), s is n int32.
 * out_rand (5n floats or NULL) receives the uniforms the ray was built from:
 * (pixel jitter u, pixel jitter v, lens disk x, lens disk y, shutter time u).                   */
int rt_generate_rays(rt_ctx* ctx, int n, int nx, int ny, const int32_t* ij, const int32_t* s,
                     uint64_t seed, float* out_origin, float* out_dir, float* out_time,
                     float* out_rand);

/* One scatter + emitted evaluation per ray with CALLER-GIVEN random inputs instead of the
 * Philox stream (shader.clj:29-119 with `rand-in-unit-sphere` = ball[3i..], `rand` = u01[i]):
 * given ray (o, d, time), hit sphere id and t, writes scattered origin/dir (3n each),
 * attenuation (3n), emitted (3n) and flags[i] = 1 if scattered, 0 if the path ends.            */
int rt_shade_batch(rt_ctx* ctx, int n, const float* origins, const float* dirs, const float* times,
                   const int32_t* hit_id, const double* hit_t, const float* ball, const float* u01,
                   float* out_origin, float* out_dir, float* out_atten, float* out_emitted,
                   int32_t* out_flags);

/* FP32 FFMA-chain peak of device 0 of the context, in TFLOP/s (2 flop per FFMA), plus the
 * packed FFMA2 figure; used as the measured roofline denominator by bench.py.                  */
int rt_measure_fp32_peak(rt_ctx* ctx, double* out_ffma_tflops, double* out_ffma2_tflops);

/* Stage profiling: when on, the wavefront variant brackets every stage kernel with CUDA events and
 * accumulates RT_CTR_{CULL,REFINE,TIEBREAK,SHADE}_NS (adds a little launch overhead; off by default). */
int rt_set_profile(rt_ctx* ctx, int on);

/* Counters accumulate over renders until reset. */
int rt_get_counters(rt_ctx* ctx, uint64_t out[RT_CTR_COUNT]);
int rt_reset_counters(rt_ctx* ctx);
int rt_device_info(rt_ctx* ctx, int* sm_count, int* clock_khz, char name[64]);

#ifdef __cplusplus
}
#endif
#endif /* RAYTRACE_B200_H */
