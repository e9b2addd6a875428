/*
 * rtp.h — C ABI of the B200 rendering core for raytracing-potato's hot path.
 *
 * This is the drop-in boundary: plain C, POD structs, borrowed pointers, status codes.
 * The reference crate (/root/reference, Rust, crate `raytracing2`) has no FFI of its own, so
 * each entry point below names the reference item it stands in for (file:line under
 * /root/reference/src). A Rust `extern "C"` block binding these symbols is shown in
 * INTEGRATION.md.
 *
 * Conventions
 *   - every function returns RTP_OK (0) or a negative rtp_status; the message for the last
 *     failure on the calling thread is available from rtp_last_error(). Nothing unwinds or
 *     aborts across this boundary (the reference panics via unwrap/assert instead).
 *   - input pointers are borrowed for the duration of the call only; the library copies what
 *     it keeps. Outputs go to caller-allocated buffers. Handles are freed by their *_destroy.
 *   - all reals are IEEE-754 binary64 (`Real = f64`, utility.rs:14). Images are row-major with
 *     row j = 0 at the BOTTOM (render.rs:66-82, image.rs:31-33).
 *   - there is no CPU fallback: every compute entry point fails with RTP_ERR_CUDA when no
 *     sm_100 device is usable.
 */
#ifndef RTP_H
#define RTP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTP_ABI_VERSION 3u

typedef enum rtp_status {
    RTP_OK = 0,
    RTP_ERR_INVALID = -1,     /* bad argument / malformed scene description           */
    RTP_ERR_IO = -2,          /* file could not be read or written (mesh.rs:145, image.rs:73) */
    RTP_ERR_FORMAT = -3,      /* unsupported TGA header / non-triangular OBJ face      */
    RTP_ERR_CUDA = -4,        /* CUDA runtime failure or no usable device              */
    RTP_ERR_NOMEM = -5,
    RTP_ERR_UNSUPPORTED = -6  /* feature outside the hot path (see DESIGN.md)          */
} rtp_status;

/* ---------------------------------------------------------------- value types ---------- */

/* utility.rs:52-57 `Ray` — 8 f64. direction is NOT required to be unit length (the reference's
 * camera produces non-unit directions, utility.rs:172-177). */
typedef struct rtp_ray {
    double origin[3];
    double direction[3];
    double t_min;
    double t_max;
} rtp_ray;

#define RTP_MISS 0xFFFFFFFFu

/* Result of one closest-hit query (bvh.rs:121-124 `Bvh::hit`, hittable.rs:110-120 `hit_list`).
 * leaf = index of the winning primitive in the hittable list handed to the scene (`LeafId`,
 * bvh.rs:9), RTP_MISS when nothing is hit; material = its MaterialId; t = `Hit::t`. */
typedef struct rtp_hit {
    uint32_t leaf;
    uint32_t material;
    double t;
} rtp_hit;

/* Full `Hit` record (utility.rs:84-89) for callers that shade on the host. */
typedef struct rtp_hit_full {
    uint32_t leaf;
    uint32_t material;
    double t;
    double position[3];
    double normal[3];
    double uv[2];
} rtp_hit_full;

/* mesh.rs:7-11 `Vertex` — 64 bytes. */
typedef struct rtp_vertex {
    double position[3];
    double normal[3];
    double uv[2];
} rtp_vertex;

/* mesh.rs:18-22 `Mesh`. indices are u32, three per face. */
typedef struct rtp_mesh {
    const rtp_vertex* vertices;
    const uint32_t* indices;
    uint32_t n_vertices;
    uint32_t n_indices;
    uint32_t material; /* MaterialId */
    uint32_t _pad;
} rtp_mesh;

/* hittable.rs:10-15 `Hittable`. The root container is expressed by rtp_scene_desc.root_kind; a container NESTED inside
 * the root's list (hittable.rs:13-14: a `List` as a BVH leaf or list item, a `Bvh` as a list item) names a run of
 * rtp_scene_desc.nested. Where the reference panics - a `Bvh` whose bounding box is needed, i.e. a `Bvh` below a `Bvh`
 * (hittable.rs:32), an empty `Bvh` (bvh.rs:40) - rtp_scene_create returns RTP_ERR_INVALID. */
typedef enum rtp_hittable_kind {
    RTP_HITTABLE_SPHERE = 0, RTP_HITTABLE_TRIANGLE = 1,
    RTP_HITTABLE_LIST = 2, /* Hittable::List(items): linear closest hit, later equal t wins (hittable.rs:110-120) */
    RTP_HITTABLE_BVH = 3   /* Hittable::Bvh(Bvh::new(items)) (bvh.rs:70-91)                                    */
} rtp_hittable_kind;

typedef struct rtp_hittable {
    uint32_t kind;     /* rtp_hittable_kind                                              */
    uint32_t material; /* sphere: MaterialId. triangle: ignored (taken from the mesh)    */
    uint32_t mesh;     /* triangle: MeshId.     list / bvh: index of its first item in rtp_scene_desc.nested */
    uint32_t triangle; /* triangle: TriangleId = index of its first entry in `indices`. list / bvh: number of items */
    double center[3];  /* sphere                                                         */
    double radius;     /* sphere                                                         */
} rtp_hittable;

/* material.rs:19-35 */
typedef enum rtp_scatter_kind {
    RTP_SCATTER_NONE = 0, RTP_SCATTER_LAMBERT = 1, RTP_SCATTER_METAL = 2, RTP_SCATTER_DIELECTRIC = 3
} rtp_scatter_kind;
/* material.rs:66-71 */
typedef enum rtp_absorb_kind {
    RTP_ABSORB_BLACKBODY = 0, RTP_ABSORB_WHITEBODY = 1, RTP_ABSORB_ALBEDO = 2, RTP_ABSORB_ALBEDO_MAP = 3
} rtp_absorb_kind;
/* material.rs:40-46 */
typedef enum rtp_emit_kind {
    RTP_EMIT_NONE = 0, RTP_EMIT_DEBUG_NORMALS = 1, RTP_EMIT_COLOR = 2, RTP_EMIT_SKY_GRADIENT = 3,
    RTP_EMIT_SKY_SPHERE = 4
} rtp_emit_kind;

/* material.rs:40-46 `Emit` (also used for the scene background, example_scenes.rs:18). */
typedef struct rtp_emit {
    uint32_t kind;   /* rtp_emit_kind        */
    uint32_t texture; /* SkySphere: TextureId */
    double rgb[3];   /* Color                */
} rtp_emit;

/* material.rs:86-91 `Material` = one scatter, one absorb, one emit. */
typedef struct rtp_material {
    uint32_t scatter;        /* rtp_scatter_kind                                   */
    uint32_t absorb;         /* rtp_absorb_kind                                    */
    uint32_t absorb_texture; /* AlbedoMap: TextureId                               */
    uint32_t _pad;
    double scatter_param;    /* Metal: fuzziness. Dielectric: refraction_index     */
    double absorb_rgb[3];    /* Albedo                                             */
    rtp_emit emit;
} rtp_material;

/* texture.rs:10-18 */
typedef enum rtp_texture_kind {
    RTP_TEXTURE_MISSING = 0, RTP_TEXTURE_DEBUG_UVS = 1, RTP_TEXTURE_SOLID = 2, RTP_TEXTURE_IMAGE = 3,
    RTP_TEXTURE_CHECKER = 4, RTP_TEXTURE_NOISE = 5, RTP_TEXTURE_PERLIN = 6
} rtp_texture_kind;

typedef struct rtp_texture {
    uint32_t kind;        /* rtp_texture_kind                                          */
    uint32_t width;       /* Image                                                     */
    uint32_t height;      /* Image                                                     */
    uint32_t odd;         /* Checker: TextureId                                        */
    uint32_t even;        /* Checker: TextureId                                        */
    uint32_t _pad;
    int64_t seed;         /* Noise / Perlin (`isize`)                                  */
    double rgb[3];        /* Solid                                                     */
    const uint8_t* rgba;  /* Image: width*height RGBA8, texel (i,j) at i + j*width,    */
                          /*        row 0 = bottom (image.rs:31-33, 92-112)            */
} rtp_texture;

typedef enum rtp_root_kind {
    RTP_ROOT_BVH = 0, /* Hittable::Bvh(Bvh::new(hittables)) — bvh.rs:70-91                */
    RTP_ROOT_LIST = 1 /* Hittable::List(hittables)          — hittable.rs:110-120         */
} rtp_root_kind;

/* render.rs:10-14 `SceneData` + example_scenes.rs:14-19 `ExampleScene` minus the camera. */
typedef struct rtp_scene_desc {
    uint32_t abi_version; /* must be RTP_ABI_VERSION */
    uint32_t root_kind;   /* rtp_root_kind           */
    const rtp_mesh* meshes;
    const rtp_hittable* hittables; /* in the order given to Bvh::new / List               */
    const rtp_material* materials;
    const rtp_texture* textures;
    uint32_t n_meshes;
    uint32_t n_hittables;
    uint32_t n_materials;
    uint32_t n_textures;
    rtp_emit background;
    const rtp_hittable* nested; /* items of nested List / Bvh hittables (may be NULL when n_nested == 0) */
    uint32_t n_nested;
    uint32_t _pad;
} rtp_scene_desc;

/* render.rs:19-25 `Camera` + utility.rs:160-163 `Transformation`.
 * orientation is the 3x3 matrix with COLUMNS x, y, z (utility.rs:176), stored column-major:
 * orientation[3*c + r] = column c, row r. */
typedef struct rtp_camera {
    double aspect_ratio;
    double fov;
    double focal_dist;
    double lens_radius;
    double orientation[9];
    double position[3];
} rtp_camera;

/* main.rs:13,25-33 renderer parameters + the work partition of main.rs:36,61-92. */
typedef struct rtp_render_params {
    uint32_t width;         /* Multisampler::width  (render.rs:58-62)                      */
    uint32_t height;        /* Multisampler::height                                        */
    uint32_t num_samples;   /* Multisampler::num_samples — the divisor (main.rs:86-87)     */
    uint32_t max_bounce;    /* depth handed to trace_path (main.rs:25, render.rs:94)       */
    uint64_t seed;          /* key of the counter-based generator that replaces StdRng     */
    uint32_t sample_begin;  /* this call traces samples [sample_begin, sample_end) of      */
    uint32_t sample_end;    /*   every pixel in the tile rectangle                         */
    uint32_t tile_x;        /* Tile::offset_i  (image.rs:143-148)                          */
    uint32_t tile_y;        /* Tile::offset_j                                              */
    uint32_t tile_w;        /* Tile::width;  0 = full frame                                */
    uint32_t tile_h;        /* Tile::height; 0 = full frame                                */
    uint32_t flags;         /* RTP_RENDER_* */
    uint32_t device_mask;   /* rtp_render / rtp_render_srgb8 on a scene made by rtp_scene_create_multi: bit d = device d takes part.
                               0 = every device of the scene. The rows of the tile rectangle are dealt out to the devices
                               round-robin and each device writes its rows straight into the host frame: no collective,
                               pixels bit-identical to a one-device render (main.rs:46-98 fans out to its workers the same way) */
    uint32_t row_offset;    /* with row_stride > 1: this call renders only rows tile_y + row_offset + k * row_stride of the    */
    uint32_t row_stride;    /*   tile rectangle (one process per GPU splitting a frame by rows); 0 or 1 = every row          */
} rtp_render_params;

#define RTP_RENDER_RAW_SUMS 1u /* write Σ over the sample range instead of Σ / num_samples   */
#define RTP_RENDER_COUNTERS 2u /* also count node visits / primitive tests (slower kernel)   */
#define RTP_RENDER_TRANSPARENT 4u /* rtp_render_srgb8: alpha = (255 * foreground) as u8 (main.rs:111,116-118) */

typedef struct rtp_stats {
    uint64_t rays;          /* closest-hit queries (`scene.hit` calls, render.rs:105,133)  */
    uint64_t paths;         /* camera samples traced                                       */
    uint64_t node_visits;   /* culling-tree nodes visited (counting kernels only)          */
    uint64_t triangle_tests;
    uint64_t sphere_tests;
    uint64_t leaf_gates;    /* exact f64 AABB::collide evaluations at leaves (bvh.rs:96)   */
    uint64_t conservative_violations; /* f32 culling decisions that contradicted the f64 test: must be 0 */
    double device_ms;       /* CUDA-event time of the device work of this call             */
    uint64_t kernel_launches;
    uint64_t order_rewalks; /* any-order walk: rays walked again in the reference's order (counting kernels only) */
    double trace_ms;        /* render calls: CUDA-event time spent in the traversal kernel launches                */
    double shade_ms;        /* render calls: ... in the generate / shade / resolve / output launches              */
} rtp_stats;

typedef struct rtp_scene_info {
    uint32_t n_leaves;
    uint32_t n_nodes;
    uint32_t depth;          /* max number of nodes on a root→leaf path */
    uint32_t root_kind;
    uint64_t device_bytes;   /* HBM held by the scene */
    uint32_t culling_depth;  /* levels of the 4-wide culling tree the kernels walk (0 for a List root)            */
    uint32_t any_order;      /* front-to-back walk: 0 = not used; rtp_scene_get_info: 1 = used, 2 = used on a scene
                                of >= 262,144 leaves (the same kernel); rtp_bvh_build_order: 1 = the scene is eligible   */
    uint32_t n_big;          /* outsized primitives exempt from distance culling (e.g. a ground sphere), at most 8 */
    uint32_t free_tree_depth;/* levels of the order-free culling tree of the any-order lanes, 0 if there is none  */
} rtp_scene_info;

typedef struct rtp_scene rtp_scene; /* opaque, immutable after creation */

/* ---------------------------------------------------------------- library --------------- */

/* Binds the calling process to `device` (one process per GPU) and creates the CUDA context.
 * Fails with RTP_ERR_CUDA if the device is missing or is not compute capability 10.x. */
int rtp_init(int device);
int rtp_device_count(int* count);
const char* rtp_last_error(void);
uint32_t rtp_abi_version(void);

/* Page-locked host memory for ray / hit / frame buffers. Buffers obtained here are copied by DMA
 * without an intermediate staging copy; ordinary malloc'd buffers are accepted everywhere too. */
int rtp_host_alloc(size_t bytes, void** out);
void rtp_host_free(void* p);

/* ---------------------------------------------------------------- assets (host) --------- */

/* mesh.rs:145-183 `obj::load`: `v`/`vn`/`vt`/`f` lines, `p/t/n` 1-based indices, vertices
 * de-duplicated by (p,t,n) in first-seen order, non-triangular faces are RTP_ERR_FORMAT,
 * material = MaterialId(0). Arrays are owned by the library; free with rtp_mesh_free. */
int rtp_obj_load(const char* path, rtp_mesh* out);
void rtp_mesh_free(rtp_mesh* mesh);

/* image.rs:11-15 `Array2d<[u8;4]>`. */
typedef struct rtp_image {
    uint8_t* rgba;
    uint32_t width;
    uint32_t height;
} rtp_image;

/* image.rs:73-114 `tga::load` (type 2, 24/32 bpp, BGR(A)→RGBA, bit-5 vertical flip) and
 * image.rs:116-137 `tga::save` (32 bpp, descriptor 0). */
int rtp_tga_load(const char* path, rtp_image* out);
int rtp_tga_save(const rtp_image* image, const char* path);
void rtp_image_free(rtp_image* image);

/* utility.rs:172-177 `Transformation::lookat`: z = normalize(position - target), x = up × z
 * (NOT normalised), y = z × x. Fills orientation and position only. */
int rtp_camera_lookat(const double position[3], const double target[3], const double up[3],
                      rtp_camera* camera);

/* utility.rs:212-220 `to_srgb_u8` over a W×H×3 f64 frame → RGBA8 (main.rs:110-122). */
int rtp_frame_to_srgb8(const double* rgb, uint32_t width, uint32_t height, uint8_t* rgba_out);

/* image.rs:151-167 `Tile::split_in_tiles`: writes up to `cap` tiles as {offset_i, offset_j,
 * width, height} quadruples in the reference's row-major order and returns their count in *n. */
int rtp_split_in_tiles(uint32_t full_width, uint32_t full_height, uint32_t tile_width,
                       uint32_t tile_height, uint32_t* tiles_out, size_t cap, size_t* n);

/* ---------------------------------------------------------------- scene ----------------- */

/* Validates and copies the description, builds the reference's median-split BVH on the host
 * (bvh.rs:36-91; centroid ties broken by LeafId, see DESIGN.md), flattens it into the device
 * node/primitive layout and uploads everything to the current device. */
int rtp_scene_create(const rtp_scene_desc* desc, rtp_scene** out);
/* The same scene replicated on every device of `device_mask` (bit d = CUDA device d; every one must be compute capability
 * 10.x). The description is flattened once and uploaded to each device. rtp_render / rtp_render_srgb8 then split a frame
 * by rows over the devices, rtp_trace_closest* / rtp_trace_camera deal their chunks out to them; the *_device entry points
 * use the first device of the mask. This is the reference's one-call-site fan-out (main.rs:46-98) across GPUs. */
int rtp_scene_create_multi(const rtp_scene_desc* desc, uint32_t device_mask, rtp_scene** out);
/* bit d set = the scene holds a replica on device d */
int rtp_scene_devices(const rtp_scene* scene, uint32_t* device_mask_out);
void rtp_scene_destroy(rtp_scene* scene);
int rtp_scene_get_info(const rtp_scene* scene, rtp_scene_info* info);
/* Leaf ids in the reference's depth-first left-to-right order (n_leaves entries). */
int rtp_scene_leaf_order(const rtp_scene* scene, uint32_t* leaf_ids_out, size_t cap);

/* Host-only half of rtp_scene_create: validates the description, runs `Bvh::new` (bvh.rs:70-91) and
 * reports the leaf ids in depth-first order plus the tree shape, without touching a device. */
int rtp_bvh_build_order(const rtp_scene_desc* desc, uint32_t* leaf_ids_out, size_t cap, rtp_scene_info* info);
/* Host-only view of the any-order walk's scene tables: the culled-set box (the union of the boxes of every primitive that is
 * not big, rounded outward to f32 as the culling tree stores boxes: min xyz, max xyz; +inf / -inf if there is none), the number
 * of leaves of the order-free culling tree and how many of them are big primitives (0 if there is no such tree). Tests only. */
int rtp_bvh_culled_set(const rtp_scene_desc* desc, float box_out[6], uint32_t* free_tree_leaves, uint32_t* free_tree_big_leaves);

/* ---------------------------------------------------------------- closest hit ----------- */

/* Batched `Hittable::hit` on the scene root (bvh.rs:121-124 / hittable.rs:110-120) for rays and
 * results in HOST memory; copies are staged through pinned buffers in chunks and overlap the
 * traversal kernel. */
int rtp_trace_closest(rtp_scene* scene, const rtp_ray* rays, size_t n, rtp_hit* hits_out,
                      rtp_stats* stats);
/* Same, plus the interpolated `Hit` fields (hittable.rs:58-62, 102-107). */
int rtp_trace_closest_full(rtp_scene* scene, const rtp_ray* rays, size_t n, rtp_hit_full* hits_out,
                           rtp_stats* stats);
/* main.rs:67-77 without the jitter: for every pixel of a width x height frame (i fastest, row j = 0 at the bottom),
 * `Camera::shoot` at the pixel centre u=(i+0.5)/W, v=(j+0.5)/H with lens_radius treated as 0 (render.rs:32-52), then
 * `Hittable::hit` on the scene root. The reference never materialises a ray array — the camera is the input of this
 * path — so rays are produced on the device and only the hits travel back to the host buffer. */
int rtp_trace_camera(rtp_scene* scene, const rtp_camera* camera, uint32_t width, uint32_t height, rtp_hit* hits_out,
                     rtp_stats* stats);
/* Same for rays/results already resident in device memory. `cuda_stream` is a cudaStream_t
 * (NULL = the legacy default stream); the call is asynchronous with respect to the host. */
int rtp_trace_closest_device(rtp_scene* scene, const rtp_ray* d_rays, size_t n, rtp_hit* d_hits_out,
                             void* cuda_stream);

/* Device-resident batch with the work counters of rtp_stats filled in (node visits, primitive
 * tests, rays, CUDA-event milliseconds). Synchronous. Used for roofline accounting. */
int rtp_trace_closest_device_counted(rtp_scene* scene, const rtp_ray* d_rays, size_t n, rtp_hit* d_hits_out,
                                     rtp_stats* stats);

/* ---------------------------------------------------------------- occlusion ------------- */

/* scene.hit(ray).is_some() (hittable.rs:18-25, bvh.rs:121-124): occluded_out[i] = 1 iff ray i hits a primitive with
 * t_min <= t <= t_max, else 0 -- bit for bit rtp_trace_closest(...).leaf != RTP_MISS. The walk stops at the first accepted leaf.
 * Host buffers, staged and dealt out over the scene's devices like rtp_trace_closest; stats as there. */
int rtp_trace_occluded(rtp_scene* scene, const rtp_ray* rays, size_t n, uint8_t* occluded_out, rtp_stats* stats);
/* scene.hit(ray).is_some() for rays/results in device memory, as rtp_trace_closest_device: asynchronous on `cuda_stream`. */
int rtp_trace_occluded_device(rtp_scene* scene, const rtp_ray* d_rays, size_t n, uint8_t* d_occluded_out, void* cuda_stream);
/* scene.hit(ray).is_some() with the work counters of rtp_stats filled in, as rtp_trace_closest_device_counted. Synchronous. */
int rtp_trace_occluded_device_counted(rtp_scene* scene, const rtp_ray* d_rays, size_t n, uint8_t* d_occluded_out, rtp_stats* stats);

/* render.rs:32-52 `Camera::shoot` for pixel-centre samples u=(i+0.5)/W, v=(j+0.5)/H of a W×H
 * frame with lens_radius treated as 0 (no random draw): writes W*H rays, i fastest, into
 * device memory. Used to build the primary-ray batch on the device. */
int rtp_camera_rays_device(const rtp_camera* camera, uint32_t width, uint32_t height,
                           rtp_ray* d_rays_out, void* cuda_stream);
/* Host-buffer convenience wrapper of the above. */
int rtp_camera_rays(const rtp_camera* camera, uint32_t width, uint32_t height, rtp_ray* rays_out);

/* ---------------------------------------------------------------- render ---------------- */

/* The worker loop of main.rs:61-92 for one tile rectangle and one sample range:
 * per pixel Σ_s trace_path(camera.shoot(jitter_s)).final_color and Σ_s hit, divided by
 * num_samples unless RTP_RENDER_RAW_SUMS. rgb_out is width*height*3 f64 (pixel (i,j) at
 * 3*(i + j*width)), foreground_out is width*height f64 (may be NULL); only pixels inside the
 * tile rectangle are written. Host buffers. */
int rtp_render(rtp_scene* scene, const rtp_camera* camera, const rtp_render_params* params,
               double* rgb_out, double* foreground_out, rtp_stats* stats);
/* rtp_render followed by the output stage of main.rs:110-122 on the device: per pixel `to_srgb_u8` (utility.rs:212-220) of
 * the averaged colour, alpha 255 or, with RTP_RENDER_TRANSPARENT, `(255 * foreground) as u8` (main.rs:116-118). rgba_out is
 * width*height*4 bytes, pixel (i,j) at 4*(i + j*width), ready for rtp_tga_save; only the tile rectangle is written.
 * The bytes equal rtp_frame_to_srgb8 of rtp_render's frame (borderline pixels are redone with the host libm). A call with
 * more than 65,536 borderline pixels among those it renders returns RTP_ERR_UNSUPPORTED (use rtp_render + rtp_frame_to_srgb8). */
int rtp_render_srgb8(rtp_scene* scene, const rtp_camera* camera, const rtp_render_params* params, uint8_t* rgba_out,
                     rtp_stats* stats);
/* Same with device output buffers; asynchronous on `cuda_stream` except for stats (pass NULL
 * stats to avoid the synchronisation). */
int rtp_render_device(rtp_scene* scene, const rtp_camera* camera, const rtp_render_params* params,
                      double* d_rgb_out, double* d_foreground_out, rtp_stats* stats,
                      void* cuda_stream);

/* ---------------------------------------------------------------- render AOVs ----------- */

/* rtp_render plus two guide buffers for a denoiser (DESIGN.md §6c). rgb_out and foreground_out hold exactly what rtp_render writes
 * for the same params. For sample s of a pixel, take the closest hit of the path's first segment (render.rs:102):
 *     A_s = the material's Absorb::evaluate at that hit (material.rs:74-81: Blackbody 0, Whitebody 1, Albedo rgb, AlbedoMap sampled
 *           at the hit's position and uv), whether or not the material scatters;
 *     N_s = Hit::normal in world space, not flipped toward the ray (a sphere's normalize(p - c), hittable.rs:60; a triangle's
 *           interpolated vertex normal, not renormalised, hittable.rs:105);
 *     both (0, 0, 0) on a miss.
 * albedo_out[3p + c] = Σ_s A_s[c] / num_samples and normal_out likewise: f64 sums from 0.0 in sample order, no contraction, the
 * colour's divisor (none with RTP_RENDER_RAW_SUMS); an averaged normal is not renormalised. Layout as rgb_out; foreground_out,
 * albedo_out and normal_out may each be NULL. Tile rectangle, rows, sample range, seed, max_bounce and device_mask as rtp_render;
 * only pixels of the tile rectangle and rows are written, and a frame split over several devices is bit-identical to one device.
 * flags must be a subset of RTP_RENDER_RAW_SUMS | RTP_RENDER_COUNTERS. stats as rtp_render. Host buffers. */
int rtp_render_aov(rtp_scene* scene, const rtp_camera* camera, const rtp_render_params* params,
                   double* rgb_out, double* foreground_out, double* albedo_out, double* normal_out, rtp_stats* stats);
/* Same with device buffers on the scene's first device; asynchronous on `cuda_stream` except for stats, as rtp_render_device. */
int rtp_render_aov_device(rtp_scene* scene, const rtp_camera* camera, const rtp_render_params* params,
                          double* d_rgb_out, double* d_foreground_out, double* d_albedo_out, double* d_normal_out,
                          rtp_stats* stats, void* cuda_stream);

/* ---------------------------------------------------------------- adaptive render ------- */

/* Stop rule of rtp_render_adaptive. */
typedef struct rtp_adaptive_params {
    uint32_t min_samples; /* samples of every pixel in round 1 (>= 1)                                       */
    uint32_t max_samples; /* no pixel takes more (>= min_samples)                                           */
    uint32_t batch;       /* samples per later round (>= 1); the last round may take fewer                   */
    uint32_t _pad;
    double abs_tol;       /* the standard error of a pixel's mean luminance must fall to abs_tol + rel_tol * |mean| */
    double rel_tol;       /*   (both finite and >= 0)                                                        */
} rtp_adaptive_params;

/* rtp_render that stops each pixel once its mean has converged (DESIGN.md §6b). The tile rectangle and rows of `params` are rendered
 * in rounds: round 1 traces samples [0, min_samples) of every pixel, each later round the next min(batch, max_samples - n) samples
 * of every pixel still live. After every round each live pixel with n samples evaluates, in f64 without contraction, over its
 * per-sample luminance Y_s = (0.2126 * r_s + 0.7152 * g_s) + 0.0722 * b_s summed in sample order from 0.0:
 *     S1 = Σ Y_s, S2 = Σ Y_s * Y_s, nd = n, mean = S1 / nd, var = (S2 - S1 * mean) / (nd - 1.0), tol = abs_tol + rel_tol * fabs(mean)
 *     stop = n >= max_samples || (n >= 2 && var / nd <= tol * tol)
 * and a pixel that stops takes no further samples (a NaN or infinite sample keeps its pixel going to max_samples).
 * With n_p the final count of pixel p: rgb_out / foreground_out hold Σ_{s < n_p} / n_p (the sums with RTP_RENDER_RAW_SUMS), bit for
 * bit rtp_render(num_samples = n_p, sample range [0, n_p)) at p; samples_out[p] = n_p (may be NULL, as may foreground_out). Layout,
 * tile, rows, seed, max_bounce and device_mask as rtp_render; only pixels of the tile rectangle and rows are written, and a frame
 * split over several devices is bit-identical to one device. params->num_samples, sample_begin and sample_end must be 0 and flags
 * a subset of RTP_RENDER_RAW_SUMS | RTP_RENDER_COUNTERS. stats->paths = Σ n_p; the other fields as rtp_render. Host buffers. */
int rtp_render_adaptive(rtp_scene* scene, const rtp_camera* camera, const rtp_render_params* params, const rtp_adaptive_params* adaptive,
                        double* rgb_out, double* foreground_out, uint32_t* samples_out, rtp_stats* stats);
/* Same with device buffers on the scene's first device. SYNCHRONOUS: every round reads one live count back, and the call returns
 * when its work on `cuda_stream` (NULL = the legacy default stream) is done. */
int rtp_render_adaptive_device(rtp_scene* scene, const rtp_camera* camera, const rtp_render_params* params, const rtp_adaptive_params* adaptive,
                               double* d_rgb_out, double* d_foreground_out, uint32_t* d_samples_out, rtp_stats* stats, void* cuda_stream);

/* ---------------------------------------------------------------- random stream --------- */

/* The counter-based generator that replaces `Randomizer = StdRng` (randomness.rs:5):
 * Philox4x32-10, key = seed, counter = (index_lo, index_hi, block, stream). Draw k of a stream
 * is word pair (k & 1) of block k >> 1, mapped to [0,1) as (u64 >> 11) * 2^-53 (the mapping of
 * rand 0.8's `Standard` for f64). Exposed so hosts and tests can reproduce device streams. */
int rtp_rng_draws(uint64_t seed, uint32_t index_lo, uint32_t index_hi, uint32_t stream,
                  uint32_t first_draw, uint32_t n_draws, double* out);

#define RTP_RNG_STREAM_PATH 0u /* (pixel j*W+i, sample s): jitter, lens, scatter draws         */
#define RTP_RNG_STREAM_RAYS 1u /* synthetic ray batches (bench / tests)                        */

/* ---------------------------------------------------------------- diagnostics ----------- */

/* Structural digests of a scene's device-resident build, read back from its first device: [0] the exact binary culling tree
 * (pre-order boxes, skip pointers, leaf slots), [1] primitive and attribute records in rank order, [2] the 4-wide culling tree
 * with its culled-set box, then the order-free culling tree if there is one, each hashed from the root down so that the numbering
 * of its nodes does not matter, [3] number of 4-wide nodes | levels << 32.
 * Two builds of the same description (host build, device build: RTP_DEVICE_BUILD) must agree in all four. Tests only. */
int rtp_scene_digest(const rtp_scene* scene, uint64_t digest_out[4]);

/* The any-order walk's scene tables as the scene holds them (DESIGN.md §4b); all zero except the empty culled-set box when the
 * scene does not take that walk. Tests only. */
typedef struct rtp_any_tables {
    uint32_t n_big;        /* outsized primitives tested before the walk, at most 8                                  */
    uint32_t big[8];       /* their slots (DFS ranks) | kind << 31, largest extent first, ties by slot; 0 past n_big  */
    uint32_t any_spheres;  /* 1: some sphere is not big                                                             */
    double any_E, any_A;   /* triangles that are not big: largest extent, largest |coordinate|, each x (1 + 1e-12)   */
    double any_C, any_R;   /* spheres that are not big: largest |box coordinate|, largest radius, each x (1 + 1e-12) */
    double scene_mag;      /* largest |coordinate| of any leaf box                                                  */
    float cull[6];         /* culled-set box: min xyz, max xyz rounded out to f32; (+inf, -inf) if empty            */
} rtp_any_tables;
int rtp_scene_any_tables(const rtp_scene* scene, rtp_any_tables* out);

/* Measured f64 instruction throughput of the bound device, in 1e9 unfused f64 operations (DMUL or DADD, the
 * only kind the path executes: the reference never contracts a*b+c) per second: the denominator of the
 * FP64 figure in bench.py's roofline (SURVEY.md 8d asks for a measured peak). Runs for a few ms. */
int rtp_probe_fp64(double* gops_out);

#ifdef __cplusplus
}
#endif
#endif /* RTP_H */
