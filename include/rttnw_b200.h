/* rttnw_b200.h — C ABI of the B200 path-tracing backend for rttnw.
 *
 * The reference (luliic2/rttnw) has NO FFI boundary: its seam is the trait
 * surface re-exported at src/math/mod.rs:10-19 plus `render` (src/main.rs:58).
 * This header is the boundary a Rust (or C++/Python) host binds instead of
 * running src/main.rs:199-229 on the CPU:
 *
 *   - the scene *description* types below are a plain-data serialisation of the
 *     reference's trait-object tree (one rtx_node per Hittable, one rtx_material
 *     per Material, one rtx_texture per Texture), so every scene the reference
 *     can express can be handed over without change of meaning;
 *   - the functions replace `World::hit` (rtx_trace_rays*), the pixel loop +
 *     `color` (rtx_render), the gamma/quantise step (rtx_tonemap_rgba8) and the
 *     nine scenes.rs constructors + scene table of main.rs (rtx_builtin_*).
 *
 * Conventions: every function returns 0 (RTX_OK) or a negative rtx_status;
 * rtx_last_error() gives the message of the last failure on the calling thread.
 * No C++ exception crosses the boundary. Handles are opaque. One rtx_ctx per
 * GPU; a ctx is used by one host thread at a time. All structs are
 * #[repr(C)]-compatible (natural alignment, explicit padding, no bitfields).
 * Nothing here falls back to the CPU: without a CUDA device every compute entry
 * point fails with RTX_ERR_CUDA.
 */
#ifndef RTTNW_B200_H
#define RTTNW_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTX_ABI_VERSION 1

typedef enum rtx_status {
    RTX_OK = 0,
    RTX_ERR_INVALID = -1, /* bad argument / malformed description */
    RTX_ERR_CUDA = -2,    /* CUDA runtime failure (incl. no device)   */
    RTX_ERR_IO = -3,      /* file could not be read / written         */
    RTX_ERR_NOMEM = -4,
    RTX_ERR_UNSUPPORTED = -5
} rtx_status;

/* ------------------------------------------------------------------ */
/* Scene description: the reference's object tree as plain data        */
/* ------------------------------------------------------------------ */

/* One entry per `impl Hittable` of src/math/hittable.rs. */
typedef enum rtx_node_kind {
    RTX_NODE_SPHERE = 1,        /* Sphere           hittable.rs:68-131  f = {cx,cy,cz,r}                    */
    RTX_NODE_MOVING_SPHERE = 2, /* MovingSphere     hittable.rs:179-245 f = {c0x,c0y,c0z,c1x,c1y,c1z,r,t0,t1} */
    RTX_NODE_RECT_XY = 3,       /* Rectangle<M,Xy>  hittable.rs:434-547 f = {a0,a1,b0,b1,k}: x in a, y in b, z=k */
    RTX_NODE_RECT_XZ = 4,       /* Rectangle<M,Xz>                      x in a, z in b, y=k                  */
    RTX_NODE_RECT_YZ = 5,       /* Rectangle<M,Yz>                      y in a, z in b, x=k                  */
    RTX_NODE_CUBE = 6,          /* Cube             hittable.rs:549-592 f = {minx,miny,minz,maxx,maxy,maxz}  */
    RTX_NODE_LIST = 7,          /* List             hittable.rs:133-177 children[child .. child+n_children)  */
    RTX_NODE_BVH = 8,           /* BvhTree::from(List) hittable.rs:247-373, same children encoding as LIST   */
    RTX_NODE_TRANSLATE = 9,     /* Translate        hittable.rs:594-629 child, f = {ox,oy,oz}                */
    RTX_NODE_ROTATE_Y = 10,     /* YRotate          hittable.rs:631-722 child, f = {angle_degrees}           */
    RTX_NODE_MEDIUM = 11        /* ConstantMedium   hittable.rs:724-801 child = boundary, f = {density},
                                   material = index of the phase-function *texture* (Isotropic albedo)     */
} rtx_node_kind;

typedef struct rtx_node {
    int32_t kind;       /* rtx_node_kind */
    int32_t material;   /* leaf geometry: material index; MEDIUM: texture index; else -1 */
    int32_t child;      /* wrapper nodes: child node index; LIST/BVH: first slot in rtx_scene_desc.children */
    int32_t n_children; /* LIST/BVH only */
    double f[10];
} rtx_node; /* 96 bytes */

/* One entry per `impl Material` of src/math/material.rs. */
typedef enum rtx_material_kind {
    RTX_MAT_LAMBERTIAN = 1,    /* material.rs:23-100   texture = albedo                     */
    RTX_MAT_METAL = 2,         /* material.rs:102-149  albedo[3], param = fuzz (<= 1)       */
    RTX_MAT_DIELECTRIC = 3,    /* material.rs:151-204  param = refraction index             */
    RTX_MAT_DIFFUSE_LIGHT = 4, /* material.rs:206-250  texture = emit                       */
    RTX_MAT_ISOTROPIC = 5      /* material.rs:252-266  texture = albedo                     */
} rtx_material_kind;

typedef struct rtx_material {
    int32_t kind;
    int32_t texture; /* texture index or -1 */
    double albedo[3];
    double param;
} rtx_material; /* 40 bytes */

/* One entry per `impl Texture` of src/math/texture.rs. */
typedef enum rtx_texture_kind {
    RTX_TEX_SOLID = 1,   /* texture.rs:9-13    f = {r,g,b}                          */
    RTX_TEX_CHECKER = 2, /* texture.rs:15-30   a = odd texture, b = even texture    */
    RTX_TEX_NOISE = 3,   /* texture.rs:32-59   a = perlin table index, f[0] = scale */
    RTX_TEX_IMAGE = 4    /* texture.rs:61-107  a = image index                      */
} rtx_texture_kind;

typedef struct rtx_texture {
    int32_t kind;
    int32_t a;
    int32_t b;
    int32_t _pad;
    double f[4];
} rtx_texture; /* 48 bytes */

/* Perlin tables (src/math/noise.rs:5-29): the reference draws them from
 * thread_rng(); here the host draws them from a seed and passes them in. */
typedef struct rtx_perlin {
    double ranvec[256][3];
    int32_t perm_x[256];
    int32_t perm_y[256];
    int32_t perm_z[256];
} rtx_perlin;

/* Decoded RGBA8 image, row 0 = top (image::RgbaImage layout, texture.rs:61-75).
 * rgba == NULL reproduces the "image failed to load" cyan texture. */
typedef struct rtx_image {
    int32_t width;
    int32_t height;
    const uint8_t* rgba;
} rtx_image;

/* CameraDescriptor, src/math/camera.rs:5-15. */
typedef struct rtx_camera {
    double lookfrom[3];
    double lookat[3];
    double view_up[3];
    double vertical_fov; /* degrees */
    double aspect_ratio;
    double aperture;
    double focus_distance;
    double open_time;
    double close_time;
} rtx_camera;

/* `struct Scene` of src/main.rs:47-55 + the object tree. All arrays are
 * borrowed for the duration of the call that receives the description. */
typedef struct rtx_scene_desc {
    const rtx_node* nodes;
    int32_t n_nodes;
    int32_t root; /* index of the world node (usually a LIST) */
    const int32_t* children;
    int32_t n_children;
    int32_t n_materials;
    const rtx_material* materials;
    const rtx_texture* textures;
    int32_t n_textures;
    int32_t n_perlins;
    const rtx_perlin* perlins;
    const rtx_image* images;
    int32_t n_images;
    int32_t _pad;
    double background[3];
    rtx_camera camera;
} rtx_scene_desc;

/* Primitive ids reported by rtx_trace_rays: a depth-first numbering of the leaf
 * primitives of the tree, starting at `root`, children in list order, a node
 * reachable twice numbered on its first visit only. SPHERE, MOVING_SPHERE and
 * RECT_* take one id; a CUBE takes six consecutive ids in the order Cube::new
 * pushes its rectangles (hittable.rs:560-569): xy(k=min.z), xy(k=max.z),
 * xz(min.y), xz(max.y), yz(min.x), yz(max.x); a MEDIUM numbers its boundary
 * subtree first and then takes one id for itself (reported on a volume hit). */
#define RTX_MISS (-1)

/* ------------------------------------------------------------------ */
/* Fixed-ray interface (replaces `world.hit(ray, t_min, t_max)`)        */
/* ------------------------------------------------------------------ */

typedef struct rtx_ray {
    double origin[3];
    double direction[3]; /* not normalised (Ray.b, src/math/ray.rs:9-13) */
    double time;         /* must lie in [min(0, camera.open_time), max(1, camera.close_time)]: the BVH bounds of a
                            MovingSphere cover its positions over that interval only (the reference's BvhTree::from uses
                            [0, 1], hittable.rs:255-258), so a ray outside it may miss a moving sphere it would hit in a
                            flat List. Render rays always comply (Camera::ray draws the time inside the shutter). */
    double t_min;
    double t_max;
    double xi; /* the uniform variate ConstantMedium::hit draws (hittable.rs:765) */
} rtx_ray;  /* 80 bytes */

/* HitRecord, src/math/hittable.rs:15-27, with the material replaced by ids. */
typedef struct rtx_hit {
    int32_t prim_id;    /* RTX_MISS when nothing was hit */
    int32_t material;   /* material index; for a medium hit: -(1 + texture index) */
    int32_t front_face; /* 0/1 */
    int32_t _pad;
    double t;
    double p[3];
    double normal[3];
    double u;
    double v;
} rtx_hit; /* 88 bytes */

/* Mean per-ray work counters of the traversal (SURVEY.md §8d: A_ray/F_ray). */
typedef struct rtx_trace_stats {
    double rays;
    double box_tests;      /* child boxes tested (2 per inner node visited)   */
    double node_visits;    /* 64-byte inner nodes fetched                      */
    double sphere_tests;   /* Sphere + MovingSphere intersection evaluations   */
    double rect_tests;
    double instance_enters; /* always 0 since wrapped primitives carry their own transform chain */
    double medium_tests;
} rtx_trace_stats;

/* ------------------------------------------------------------------ */
/* Render interface (replaces src/main.rs:199-229 and :26-45)           */
/* ------------------------------------------------------------------ */

typedef struct rtx_render_params {
    int32_t width;
    int32_t height;
    int32_t spp_begin; /* first global sample index rendered by this call  */
    int32_t spp_count; /* number of samples per pixel rendered by this call */
    int32_t max_depth; /* 50 in the reference (src/main.rs:216)             */
    int32_t _pad;
    uint64_t seed;     /* Philox key; identical images for identical seeds  */
} rtx_render_params;

typedef struct rtx_ctx rtx_ctx;
typedef struct rtx_scene rtx_scene;

/* ---- library ---- */
int rtx_abi_version(void);
const char* rtx_last_error(void);
int rtx_device_count(int* count);

/* ---- context: one per GPU. `stream` is a cudaStream_t to launch on (e.g. the
 * caller's torch stream) or NULL to let the context create its own non-blocking
 * stream. To launch on the default stream pass the explicit handles
 * cudaStreamLegacy ((void*)0x1) or cudaStreamPerThread ((void*)0x2). ---- */
int rtx_ctx_create(int device, void* stream, rtx_ctx** out);
int rtx_ctx_destroy(rtx_ctx* ctx);
int rtx_ctx_sync(rtx_ctx* ctx);
/* Asynchronous rendering (off by default). The wavefront driver behind rtx_render feeds the stream in batches and
 * watches a completion counter, which keeps the calling thread busy for the length of the render. With on != 0 that
 * loop runs on a thread the context owns: rtx_render queues the job and returns at once (the parameter struct is
 * copied; scene and accumulator must stay alive), so one host thread can keep several GPUs rendering. Every other
 * entry point taking this ctx — rtx_ctx_sync above all — first waits for that thread to run dry, which keeps the
 * calls of ONE context in program order; an asynchronous render that failed reports its error from the next such
 * call. Work the caller puts on the ctx stream BEHIND the ABI's back (e.g. torch ops on a shared stream) is not
 * ordered against a queued render: call rtx_ctx_sync first. Destroy a scene only after syncing the contexts that
 * render it. */
int rtx_ctx_set_async(rtx_ctx* ctx, int on);
void* rtx_ctx_stream(rtx_ctx* ctx);
/* Which builder makes the BVH over the world in rtx_scene_create (replaces BvhTree::new, hittable.rs:260-321; the
 * tree's topology is not part of the contract, only the closest-hit answers): 0 = host, binned SAH (default, the
 * better trees), 1 = device, Morton-code LBVH, 2 = device, PLOC (locally-ordered agglomerative clustering along the Morton
 * curve: merges decided by box surface areas), 3 = device, top-down binned SAH (the host builder's policy: trees of
 * host quality) — the device builders are for scenes large enough that the host build is the bottleneck. Other kinds
 * are refused. */
int rtx_ctx_set_bvh_builder(rtx_ctx* ctx, int kind);
/* number of CUDA kernels this context has launched so far (bookkeeping for benchmarks) */
int rtx_ctx_kernel_launches(rtx_ctx* ctx, unsigned long long* out);
/* Per-kernel timing of rtx_render (benchmark bookkeeping): when on, the shade / trace launches of
 * every 8th iteration are bracketed by CUDA events on the ctx stream (scaled back up by 8) and
 * rtx_render waits for the last one before it returns. rtx_ctx_profile_read returns the accumulated device milliseconds of the two kernels and
 * the number of (shade, trace) iterations they cover; reset != 0 clears the accumulators. */
int rtx_ctx_set_profiling(rtx_ctx* ctx, int on);
int rtx_ctx_profile_read(rtx_ctx* ctx, double* shade_ms, double* trace_ms,
                         unsigned long long* iterations, int reset);
/* Roofline denominator for this path (benchmark bookkeeping): the flattened scene and the path pool live in L2,
 * so the bandwidth that bounds BVH-node traffic is L2's, not HBM's. Reads an L2-resident buffer of `bytes`
 * (0 = 32 MiB) `repeats` times (0 = 64) with 16-byte loads that skip L1 from every SM and reports GB/s. */
int rtx_ctx_measure_l2_read(rtx_ctx* ctx, unsigned long long bytes, int repeats, double* gbytes_per_s);

/* ---- scene: flattens the tree, builds the BVHs, uploads (host memory is
 * copied; the caller keeps ownership of everything in `desc`). ---- */
int rtx_scene_create(rtx_ctx* ctx, const rtx_scene_desc* desc, rtx_scene** out);
int rtx_scene_destroy(rtx_scene* scene);
/* rtx_scene_destroy keeps up to four device arenas / texture arrays per device for the next rtx_scene_create (a host
 * that re-uploads its scene every frame then pays two copies instead of cudaMalloc + cudaFree): this frees them. */
int rtx_cache_trim(int device);
/* sizes of the flattened device representation (for roofline bookkeeping) */
int rtx_scene_info(const rtx_scene* scene, int32_t* n_bvh_nodes, int32_t* n_records,
                   int32_t* n_xform_ops, int64_t* device_bytes);

/* ---- fixed rays ---- */
/* host buffers: H2D, kernel, D2H, synchronous */
int rtx_trace_rays(rtx_ctx* ctx, const rtx_scene* scene, int64_t n, const rtx_ray* rays,
                   rtx_hit* hits);
/* device buffers: asynchronous on the ctx stream */
int rtx_trace_rays_device(rtx_ctx* ctx, const rtx_scene* scene, int64_t n,
                          const rtx_ray* d_rays, rtx_hit* d_hits);
/* counting variant (device buffers, synchronous): mean work per ray */
int rtx_trace_rays_stats(rtx_ctx* ctx, const rtx_scene* scene, int64_t n, const rtx_ray* d_rays,
                         rtx_trace_stats* out);

/* ---- render ---- */
/* Adds spp_count samples per pixel into d_accum (device, width*height float4:
 * sum r, sum g, sum b, sample count; row 0 = TOP row, matching the order the
 * reference emits pixels, src/main.rs:202-204). All work is ordered on the ctx
 * stream and the result is NOT synchronised on return. By default the call keeps
 * the calling thread busy while it feeds the stream (the wavefront driver polls
 * a completion counter); after rtx_ctx_set_async(ctx, 1) it returns at once. Samples are added with atomics: the fp32 summation
 * order, hence the last bits of the sums, can differ from run to run.
 * d_ray_count (device uint64, may be NULL) is incremented by the number of
 * world.hit queries issued. The sample count of a pixel is kept in the fp32 .w of
 * the accumulator: at most 2^24 samples per pixel can be accumulated in one
 * buffer (16.7 M; the reference's largest default is 10^4), and at most 2^24 per
 * call. Uniform variates are 24-bit (word >> 8) / 2^24: exact in fp32 and f64
 * alike, which is what makes accept / reject decisions identical to the
 * oracle's; a ConstantMedium therefore never samples a free flight longer than
 * 24 ln 2 / density (16.6 mean free paths), where the reference's 53-bit draws
 * reach 36.7. */
int rtx_render(rtx_ctx* ctx, const rtx_scene* scene, const rtx_render_params* params,
               float* d_accum, unsigned long long* d_ray_count);
/* Same render through the counting build of the kernel (slower; for roofline bookkeeping):
 * synchronous, returns the number of world.hit queries in out->rays and the MEAN work per
 * query in the other fields. */
int rtx_render_counted(rtx_ctx* ctx, const rtx_scene* scene, const rtx_render_params* params,
                       float* d_accum, rtx_trace_stats* out);
/* mean, sqrt gamma, clamp(0,0.999)*256 -> u8, alpha 255 (src/main.rs:217-225).
 * d_accum: device float4 per pixel. out: RGBA8, host (out_on_device=0,
 * synchronous) or device (asynchronous). */
int rtx_tonemap_rgba8(rtx_ctx* ctx, const float* d_accum, int32_t width, int32_t height,
                      uint8_t* out, int out_on_device);
/* Adaptive sampling. The reference gives every pixel the same number of samples (the fixed per-pixel fold of
 * src/main.rs:211); here each 8x4 tile of pixels stops once its noise estimate is below a threshold. Every pixel ends
 * with the samples [spp_begin, spp_begin + n) of the uniform render (a prefix of its sample sequence), n shared by the
 * pixels of a tile: round 0 renders min_spp samples for every tile, each later round min(step_spp, max_spp - n) more
 * for the tiles still sampling. d_aux (width*height float4, like d_accum) receives only the samples with an odd
 * global index, so aux.w == n / 2. The pixel error compares the two halves' means I = accum.rgb / accum.w and
 * A = aux.rgb / aux.w, with the sqrt gamma of main.rs:217-225 in the denominator:
 *     e = (|I_r - A_r| + |I_g - A_g| + |I_b - A_b|) / (1e-4 + sqrt(I_r + I_g + I_b)),
 * a tile's error is the largest e of its pixels inside the frame (a pixel with no samples in either buffer counts 0),
 * and after each round a tile whose error is below the threshold stops for good, as does every tile at max_spp. */
typedef struct rtx_adaptive_params {
    double threshold; /* >= 0, finite; 0 = every pixel gets max_spp (params->spp_count) */
    int32_t min_spp;  /* even, >= 2, <= max_spp */
    int32_t step_spp; /* even, >= 2 */
} rtx_adaptive_params; /* 16 bytes */

typedef struct rtx_adaptive_stats {
    int64_t path_samples;    /* sum of n over the pixels of the frame */
    int32_t rounds;          /* render rounds */
    int32_t tiles;           /* 8x4 tiles of the frame */
    int32_t tiles_converged; /* stopped below the threshold before max_spp */
    int32_t tiles_at_max;    /* stopped at max_spp (tiles_converged + tiles_at_max == tiles) */
} rtx_adaptive_stats; /* 24 bytes */

/* params->spp_count is max_spp (even, <= 2^24); params->spp_begin is even. Zeroes d_accum and d_aux, then renders.
 * Synchronous: joins any queued asynchronous job first (like rtx_render_counted). stats may be NULL. Needs the
 * default wavefront driver: RTX_MODE=mega, RTX_SHADE=1 and RTX_ORDER=1 give RTX_ERR_UNSUPPORTED. */
int rtx_render_adaptive(rtx_ctx* ctx, const rtx_scene* scene, const rtx_render_params* params,
                        const rtx_adaptive_params* adaptive, float* d_accum, float* d_aux,
                        rtx_adaptive_stats* stats);
/* Per-tile error of any (accum, aux) pair: tiles_y x tiles_x floats, row 0 = top tiles. Asynchronous.
 * This is the same error rtx_render_adaptive decides on, so a user can show a noise map. */
int rtx_adaptive_error(rtx_ctx* ctx, const float* d_accum, const float* d_aux, int32_t width, int32_t height,
                       float* d_tile_error);
/* Feature buffers ("AOVs") of the first vertex of every path, for denoisers and compositors. For every pixel and every
 * global sample index s in [spp_begin, spp_begin + spp_count), take the path rtx_render follows for (pixel, s) with the
 * same seed: the same camera ray (jitter, lens, shutter time) and the same bounce-0 draws, each ConstantMedium's
 * free-flight draw included. Its first vertex is the closest of the surface hit and any medium scatter point in front
 * of it, exactly as the render's bounce 0 decides. Per sample the call adds (layouts width*height, row 0 = top, like
 * d_accum):
 *   d_albedo  float4 {sum r, sum g, sum b, n}: Lambertian / Isotropic: the texture value at the vertex; Metal: its
 *             albedo, whether or not the scatter is absorbed; Dielectric: (1, 1, 1), the reference's attenuation;
 *             DiffuseLight: its emitted texture value clamped to [0, 1]; a miss: the background clamped to [0, 1].
 *   d_normal  float4 {sum nx, sum ny, sum nz, n}: the hit record's normal as the render uses it (front-face oriented,
 *             hittable.rs:30-44); 0 for a medium vertex (whose normal is arbitrary in the reference) and for a miss.
 *   d_depth   float2 {sum dist, hits}: dist = t * |d|, the distance from the ray's origin on the lens to the vertex;
 *             only samples that have a vertex add, and `hits` counts them.
 * The call ADDS into the buffers, so chunked calls compose; a buffer pointer may be NULL (not wanted), all three NULL
 * is RTX_ERR_INVALID. params is validated like rtx_render's; max_depth must be >= 1 and does not matter otherwise.
 * Asynchronous on the ctx stream; joins any queued asynchronous job first. Deterministic: each pixel sums its samples
 * in ascending order in registers and adds the sums once (one thread per pixel, no atomics), so a call's result is
 * bit-identical from run to run. The samples are keyed like the beauty's: a pass over [0, k) describes the same
 * paths as the first k samples of a render. */
int rtx_render_aov(rtx_ctx* ctx, const rtx_scene* scene, const rtx_render_params* params, float* d_albedo,
                   float* d_normal, float* d_depth);
/* Denoiser: an edge-avoiding à-trous wavelet filter (Dammertz et al., HPG 2010) steered by a per-pixel variance
 * estimate (as in SVGF, Schied et al., HPG 2017), over the beauty and the feature buffers. All buffers are device
 * memory, width*height float4, row 0 = top: d_accum as rtx_render fills it; d_half a subset of the same samples chosen
 * without looking at their values (the d_aux of rtx_render_adaptive, or the accumulator copied with rtx_memcpy_d2d
 * between the renders of [0, n/2) and [n/2, n)); d_albedo and d_normal as rtx_render_aov fills them. d_out receives
 * {r, g, b, 1}, which rtx_tonemap_rgba8 and rtx_pfm_write (after dropping .w) take unchanged.
 * Per pixel p, with L(x) = 0.2126 x.r + 0.7152 x.g + 0.0722 x.b:
 *   n = accum.w, m = half.w; a pixel with n == 0 has no samples: it contributes nothing and outputs {0, 0, 0, 1}.
 *   c = accum.rgb / n;  a = albedo.rgb / albedo.w (0 if albedo.w == 0);  a' = max(a, 1e-3) per channel;
 *   N = normal.xyz / normal.w (0 if normal.w == 0), not renormalised (0 at medium vertices and misses);
 *   e = c / a' (demodulated irradiance);
 *   v = L((H - R) / a')^2 * m (n - m) / n^2 if 0 < m < n, else 0, where H = half.rgb / m, R = (accum.rgb - half.rgb) /
 *       (n - m): since E[(H - R)^2] = sigma^2 n / (m (n - m)), v estimates the variance of the mean, sigma^2 / n.
 * Pass i = 0 .. iterations-1, step s = 2^i, over the pixels with samples:
 *   g_p = sum k v_q / sum k over the 3x3 neighbours q (step 1) in the frame with samples, k = [1/4, 1/2, 1/4] per axis;
 *   for the taps q = p + s (dx, dy), dx, dy in -2..2, in the frame and with samples, with h = [1, 4, 6, 4, 1] / 16:
 *     w = h(dx) h(dy) exp(-|N_p - N_q|^2 / sigma_normal^2 - |a_p - a_q|^2 / sigma_albedo^2
 *                         - |L(e_p) - L(e_q)| / (sigma_luminance sqrt(g_p) + 1e-10));
 *   e_p <- sum w e_q / sum w,  v_p <- sum w^2 v_q / (sum w)^2  (all pixels update from the previous pass's values).
 * Output: out_p = {e_p a'_p, 1}. Depth is deliberately not a weight: at a medium vertex it is a free-flight draw.
 * The output is BIASED, unlike every other output of the library: a filtered estimate, not a sample mean.
 * Asynchronous on the ctx stream; joins any queued asynchronous job first. Deterministic (one thread per pixel, no
 * atomics): bit-identical from run to run. The inputs are not modified. RTX_ERR_INVALID: a NULL or not 16-byte
 * aligned buffer (the kernels load and store float4), a d_out that overlaps an input, a size <= 0 or of 2^31 pixels or
 * more, iterations outside [1, 10], a sigma <= 0 or not finite, and a sigma_normal or sigma_albedo below about 5.4e-20
 * (the kernels multiply by 1 / sigma^2 in fp32, which must be finite). Any width and height within 2^31 pixels are
 * accepted. The context keeps 56 bytes a pixel of scratch, grown as needed. params == NULL takes the defaults below. */
typedef struct rtx_denoise_params {
    int32_t iterations;    /* à-trous passes, in [1, 10]; pass i takes taps 2^i pixels apart (default 5) */
    float sigma_normal;    /* > 0, finite (default 0.25) */
    float sigma_albedo;    /* > 0, finite (default 0.1) */
    float sigma_luminance; /* > 0, finite (default 8) */
} rtx_denoise_params;      /* 16 bytes */
int rtx_denoise(rtx_ctx* ctx, const float* d_accum, const float* d_half, const float* d_albedo, const float* d_normal,
                int32_t width, int32_t height, const rtx_denoise_params* params, float* d_out);
/* Rank-0 side of the multi-GPU combine: sums n_peers device accumulators
 * (peer-mapped pointers, read over NVLink) into d_accum and tonemaps in the
 * same kernel. d_rgba8 is a device buffer. Asynchronous. DESTRUCTIVE: d_accum
 * receives the sum (so that rank 0 can checkpoint or keep accumulating the
 * combined frame) — call it once per frame, a second call would add the peers
 * again. A peer on a device this one cannot map (no NVLink / PCIe peer-to-peer)
 * is staged through a scratch buffer with cudaMemcpyPeerAsync instead. */
int rtx_reduce_tonemap_peers(rtx_ctx* ctx, float* d_accum, const float* const* d_peer_accums,
                             int32_t n_peers, int32_t width, int32_t height, uint8_t* d_rgba8);

/* The same combine with the work spread over the ranks: EVERY rank calls this with the accumulators of all n_ranks
 * ranks (its own and the peer-mapped / IPC-opened others, in rank order) and reduces + tonemaps pixels
 * [rank * n / n_ranks, (rank + 1) * n / n_ranks) only, writing them straight into rank 0's RGBA8 buffer
 * (d_rgba8_root: local on rank 0, peer-mapped elsewhere). Nothing is written back to the accumulators, so unlike
 * rtx_reduce_tonemap_peers it can be repeated. The caller orders the ranks (a barrier before and after). */
int rtx_reduce_tonemap_slice(rtx_ctx* ctx, const float* const* d_accums, int32_t n_ranks, int32_t rank,
                             int32_t width, int32_t height, uint8_t* d_rgba8_root);
/* NCCL form of the combine (SURVEY.md §8b: the fold of src/main.rs:211-217 across ranks as one
 * ncclReduce(sum, float, width*height*4) to `root`, in place, on the ctx stream; follow it with rtx_tonemap_rgba8 on
 * the root). libnccl.so.2 is opened at the first call — RTX_ERR_UNSUPPORTED when the host has none. One rank makes
 * the 128-byte id and hands it to the others by whatever channel the host has (a pipe, MPI, torch.distributed);
 * rtx_comm_create is collective over the n_ranks contexts. rtx_comm_wrap adopts an ncclComm_t the host already owns. */
typedef struct rtx_comm rtx_comm;
int rtx_comm_unique_id(uint8_t id_out[128]);
int rtx_comm_create(rtx_ctx* ctx, int32_t n_ranks, int32_t rank, const uint8_t id[128], rtx_comm** out);
int rtx_comm_wrap(void* nccl_comm, rtx_comm** out);
int rtx_comm_destroy(rtx_comm* comm);
int rtx_accum_reduce(rtx_ctx* ctx, rtx_comm* comm, float* d_accum, int32_t width, int32_t height, int32_t root);

/* ---- device memory + CUDA IPC helpers so that a non-torch host (the Rust
 * crate, the C++ CLI) can drive everything through this ABI alone ---- */
int rtx_malloc(rtx_ctx* ctx, size_t bytes, void** out);
int rtx_free(rtx_ctx* ctx, void* ptr);
int rtx_memset_zero(rtx_ctx* ctx, void* ptr, size_t bytes);
int rtx_memcpy_h2d(rtx_ctx* ctx, void* dst, const void* src, size_t bytes);
int rtx_memcpy_d2h(rtx_ctx* ctx, void* dst, const void* src, size_t bytes);
/* device to device, asynchronous on the ctx stream (e.g. the d_half of rtx_denoise) */
int rtx_memcpy_d2d(rtx_ctx* ctx, void* dst, const void* src, size_t bytes);
int rtx_ipc_export(rtx_ctx* ctx, void* d_ptr, uint8_t handle_out[64]);
int rtx_ipc_open(rtx_ctx* ctx, const uint8_t handle[64], void** d_ptr_out);
int rtx_ipc_close(rtx_ctx* ctx, void* d_ptr);

/* ------------------------------------------------------------------ */
/* Host-side mirrors of scenes.rs / main.rs (no GPU needed)             */
/* ------------------------------------------------------------------ */

/* The scene table of src/main.rs:66-183 + defaults of :255. */
typedef struct rtx_scene_defaults {
    int32_t width;
    int32_t height;
    int32_t samples;
    int32_t max_depth;
    const char* name;
} rtx_scene_defaults;
int rtx_builtin_scene_defaults(int scene_number, rtx_scene_defaults* out);

/* Builds scene 1..9 (scenes.rs:11-334). The reference draws geometry, Perlin
 * tables etc. from thread_rng(); here they come from SplitMix64(seed).
 * `earth_png_path` is the file ImageTexture::new opens (scenes.rs:129,303);
 * NULL means "assets/earth.png" relative to the CWD like the reference; an
 * unreadable file gives the cyan texture (texture.rs:96-99), not an error. */
int rtx_builtin_scene(int scene_number, uint64_t seed, const char* earth_png_path,
                      rtx_scene_desc** out);
int rtx_scene_desc_free(rtx_scene_desc* desc);

/* Host-only self check of the flattening step (no GPU): flattens `desc`, builds
 * the BVHs and verifies that every record lies inside every ancestor box and is
 * reachable exactly once. Outputs may be NULL. */
int rtx_flatten_check(const rtx_scene_desc* desc, int32_t* n_bvh_nodes, int32_t* n_records,
                      int32_t* n_prim_ids);

/* PNG I/O (zlib based): 8-bit gray/RGB/RGBA(+alpha) non-interlaced decode to
 * RGBA8, RGBA8 encode (image::save_buffer, src/main.rs:231). */
int rtx_png_read_rgba8(const char* path, int32_t* width, int32_t* height, uint8_t** rgba_out);
int rtx_png_write_rgba8(const char* path, int32_t width, int32_t height, const uint8_t* rgba);
/* PFM (portable float map) writer for linear images: channels 3 ("PF") or 1 ("Pf"), anything else is
 * RTX_ERR_INVALID. `data` is host memory, width*height*channels floats, row 0 = top; the file stores the rows
 * bottom-up as little-endian floats (scale -1.0). */
int rtx_pfm_write(const char* path, int32_t width, int32_t height, int32_t channels, const float* data);
int rtx_buffer_free(void* p);

#ifdef __cplusplus
}
#endif
#endif /* RTTNW_B200_H */
