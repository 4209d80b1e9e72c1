/*
 * fspt_b200.h -- C ABI of libfspt_b200.so: the B200 (sm_100a) replacement for the GPU hot path of
 * apbodnar/FSPT (camera.fs -> tracer.fs / bvh_test.fs -> draw.fs, driven by main.js).
 *
 * The reference has no FFI; its de-facto operator surface is the set of GL resources, #defines and
 * uniforms main.js hands to its three programs.  Every entry point below names the reference
 * interface it replaces (file:line relative to the reference root).  See INTEGRATION.md for the
 * N-API / ctypes bindings a maintainer would add.
 *
 * Conventions
 *  - every call returns 0 on success, a negative FSPT_E_* code otherwise; fspt_last_error() gives text
 *    (the reference logs shader errors and returns null, main.js:91-94, or throws a string, :564-569);
 *  - all input pointers are HOST pointers, borrowed for the duration of the call only (texImage2D/3D copy
 *    typed arrays synchronously, main.js:412-437,557-559); the library owns all device memory;
 *  - one context is used by one host thread at a time (the reference is a single JS thread);
 *  - images are in GL order: index = y*width + x with y = 0 the BOTTOM row (gl_FragCoord / readPixels).
 *  - there is NO CPU fallback: every call fails with FSPT_E_CUDA when no sm_100 device is present.
 */
#ifndef FSPT_B200_H
#define FSPT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FSPT_ABI_VERSION 3

enum {
  FSPT_OK = 0,
  FSPT_E_INVALID = -1, /* bad argument / malformed scene buffers */
  FSPT_E_CUDA = -2,    /* CUDA runtime error, or no usable device */
  FSPT_E_STATE = -3,   /* call out of order (e.g. render before scene upload) */
  FSPT_E_LIMIT = -4,   /* scene exceeds a documented limit (BVH deeper than the traversal stack) */
  FSPT_E_NCCL = -5     /* NCCL could not be loaded, or a collective failed */
};

typedef struct fspt_ctx fspt_ctx;

/* Static scene inputs == the data textures + atlas + env + bins + #defines built by initBVH()
 * (main.js:284-445), un-padded (padBuffer's -1 fill, main.js:143-154, is a texture artefact that the
 * library re-creates as LEAF_SIZE-1 degenerate tail triangles). */
typedef struct fspt_scene_desc {
  const float* bvh;        /* bvhBuffer after maskBVHBuffer: 9 f32/node, [left,right,triIndex] are int32 bits
                              (main.js:366-392,272-282); node 0 = root                                  */
  const float* triangles;  /* trianglesBuffer: 9 f32/tri, leaf order (main.js:374)                      */
  const float* materials;  /* materialBuffer: 12 f32/tri (main.js:377-382)                              */
  const float* normals;    /* normalBuffer: 27 f32/tri, [n,t,b] per vertex (main.js:383-385)            */
  const float* uvs;        /* uvBuffer: 6 f32/tri (main.js:386)                                         */
  const float* lights;     /* lightBuffer: 9 f32/light-tri (main.js:394-401); accepted, unused by
                              tracer.fs main() (dead code in the reference), may be NULL                */
  const float* light_ranges; /* lightRanges pairs (main.js:395,400); may be NULL                        */
  const uint8_t* atlas;    /* TexturePacker.getPixels(): res*res*4*layers bytes (main.js:556-559)       */
  const uint8_t* env;      /* RGBE-in-RGBA8 environment, row 0 = image top (main.js:170-180)            */
  const uint16_t* radiance_bins; /* ProcessEnvRadiance(): [x0,y0,x1,y1] per bin (main.js:298-299)       */
  int32_t n_nodes;
  int32_t n_triangles;
  int32_t n_light_triangles;
  int32_t n_light_ranges;  /* '#define NUM_LIGHT_RANGES' (main.js:402-406)                              */
  int32_t atlas_res;       /* texturePacker.setAndGetResolution() (main.js:556)                         */
  int32_t atlas_layers;    /* texturePacker.imageSet.length                                             */
  int32_t env_width, env_height;
  int32_t env_bins;        /* '#define ENV_BINS' (main.js:299)                                          */
  int32_t leaf_size;       /* '#define LEAF_SIZE' (main.js:895); must be 4 (kernels are specialised)    */
} fspt_scene_desc;

/* Per-frame uniforms of drawCamera() (main.js:741-756) and drawTracer() (main.js:758-807). */
typedef struct fspt_frame_params {
  float eye[3];            /* uniform P (main.js:751)                    */
  float dir[3];            /* uniform I (main.js:752), used un-normalised */
  float fov_scale;         /* main.js:747                                */
  float lens_features[2];  /* [1 - 1/focalDepth, aperture] (main.js:749) */
  float env_theta;         /* main.js:778, in turns                      */
} fspt_frame_params;

/* Uniforms of drawQuad() (main.js:809-824). */
typedef struct fspt_post_params {
  float exposure, saturation, max_sigma, scale;
  int32_t denoise;
} fspt_post_params;

typedef struct fspt_stats {
  uint64_t samples;       /* path samples rendered since fspt_clear (pixels * ticks; with adaptive sampling,
                             the samples of the active pixels, counted on the device)                 */
  uint64_t rays;          /* intersectScene-equivalent calls: primary + shadow + continuation        */
  uint64_t node_visits;   /* V: loop iterations of intersectScene (tracer.fs:373)                    */
  uint64_t leaf_visits;   /* L: processLeaf calls (tracer.fs:380)                                    */
  uint64_t kernel_launches;
  double trace_ms;        /* CUDA-event time spent in traversal kernels during the last fspt_render  */
  double render_ms;       /* CUDA-event time of the last fspt_render (camera+trace+shade+accumulate) */
  uint64_t last_rays, last_node_visits, last_leaf_visits; /* of the last fspt_render only            */
  uint64_t capped_paths;  /* paths stopped by the refraction safety cap                              */
  double shade_ms;        /* CUDA-event time spent in shading kernels during the last fspt_render    */
  double reduce_ms;       /* CUDA-event time of the last fspt_reduce_accum (NCCL reduce on the context's stream) */
  double primary_trace_ms; /* part of trace_ms spent in the camera + primary-ray launches (camera.fs + the first
                              intersectScene of tracer.fs main, :440) of the last fspt_render */
  /* trace_ms, shade_ms and primary_trace_ms are sums of per-launch event times.  A large wave is rendered as two
   * row bands on two streams whose launches overlap, so trace_ms + shade_ms can exceed render_ms; render_ms is the
   * wall time of the render on the device. */
} fspt_stats;

int fspt_abi_version(void);

/* initGL()+initBuffers() (main.js:77-85,598-617): canvas size, the two RGBA32F screen targets and the
 * camera pos/dir targets.  device = CUDA ordinal. */
int fspt_create(fspt_ctx** out, int32_t width, int32_t height, int32_t device);
void fspt_destroy(fspt_ctx* ctx);
const char* fspt_last_error(const fspt_ctx* ctx); /* ctx may be NULL: error of the failed fspt_create */

/* The texImage2D/3D uploads of initBVH()/initAtlas() (main.js:408-437,548-560,170-180). */
int fspt_scene_upload(fspt_ctx* ctx, const fspt_scene_desc* scene);
/* The same upload, returning as soon as every buffer EXCEPT scene->atlas has been consumed (texImage3D of the atlas,
 * main.js:556-559, is by far the largest transfer and only the shading pass reads it): the atlas is staged and DMA'd
 * by a thread of the context while the caller goes on -- typically into fspt_render, whose camera + primary traversal
 * launch then overlaps the atlas transfer; the library waits for the staging itself before its first shading launch.
 * scene->atlas -- and scene->env when it is page-locked, see fspt_host_register -- must stay valid and unchanged until
 * fspt_scene_upload_wait (or fspt_synchronize, the next upload, or fspt_destroy) has returned; errors of the staging are
 * reported by whichever call joins it. */
int fspt_scene_upload_async(fspt_ctx* ctx, const fspt_scene_desc* scene);
int fspt_scene_upload_wait(fspt_ctx* ctx);
/* Optional: page-lock a host buffer the caller keeps across uploads (cudaHostRegister; no reference counterpart --
 * WebGL copies out of JS memory).  fspt_scene_upload(_async) recognises page-locked memory by itself, whoever locked it:
 * a page-locked `atlas` is DMA'd from where it lies (only its distinct non-constant layers cross PCIe; the per-material
 * texels are built on the GPU) and a page-locked `env` likewise; the geometry buffers are always repacked through the
 * library's own staging.  Errors of these two calls are reported through fspt_last_error(NULL). */
int fspt_host_register(void* ptr, uint64_t bytes);
int fspt_host_unregister(void* ptr);

/* clear() (main.js:826-836): zero the accumulation target, pingpong = 0. */
int fspt_clear(fspt_ctx* ctx);

/* n_samples iterations of { drawCamera(); drawTracer(tick) } (main.js:841-845), tick = first_tick + k.
 * rand_base_camera[k] / rand_base_tracer[k] are the two `Math.random()*10000` uniforms of iteration k
 * (main.js:748,777), supplied by the host so that runs are reproducible.  Asynchronous: kernels are
 * enqueued on the context's stream; fspt_resolve / fspt_read_* / fspt_stats synchronise. */
int fspt_render(fspt_ctx* ctx, const fspt_frame_params* frame, uint32_t first_tick, int32_t n_samples,
                const float* rand_base_camera, const float* rand_base_tracer);

/* drawQuad() (main.js:809-824, draw.fs): firefly filter, exposure, ACES, saturation, gamma -> RGBA8,
 * width*height*4 bytes, GL row order (what readPixels / toBlob sees, main.js:861). */
int fspt_resolve(fspt_ctx* ctx, const fspt_post_params* post, uint8_t* rgba8_out);

/* Accumulation target textures.screen[pingpong%2] (RGBA32F, main.js:575,608-610); never read back by the
 * reference, exposed for parity tests, checkpoint/resume and multi-GPU merging. */
int fspt_read_accum(fspt_ctx* ctx, float* rgba32f_out);
int fspt_write_accum(fspt_ctx* ctx, const float* rgba32f_in, uint32_t next_tick);

/* Accumulation mode: 0 = the reference's running mean (tracer.fs:517), bit-faithful, default;
 * 1 = plain f32 sum, with every pixel's sample count in the alpha channel (what tile / sample-set sharding across
 * GPUs reduces with NCCL); fspt_resolve then divides each pixel by its own count. */
int fspt_set_accum_mode(fspt_ctx* ctx, int32_t mode);
/* Device pointer + element count (floats) of the accumulation buffer and the number of samples summed
 * into it, for torch.distributed / NCCL reduction by the host.  The pointer stays valid until destroy. */
int fspt_accum_device_ptr(fspt_ctx* ctx, void** dptr, uint64_t* n_floats, uint64_t* n_samples);
int fspt_set_accum_samples(fspt_ctx* ctx, uint64_t n_samples);

/* ---- adaptive sampling (sum mode only; no reference counterpart) -------------------------------------------------
 * max_rel_error > 0 turns it on for later fspt_render calls, 0 turns it off (the default).  FSPT_E_INVALID for a NaN or
 * negative max_rel_error or for min_samples < 2 (a variance needs two samples).  While it is on, fspt_render in
 * accumulation mode 0 returns FSPT_E_STATE: the running mean keeps no per-pixel count.
 * Before each wave of a render, every pixel of the context's rectangle is tested; an ACTIVE pixel gets all samples of
 * the wave, the others none.  With n = the pixel's count (alpha), m2 = its moment (below), every step in f32, in order:
 *   mean   = ((r*0.2126 + g*0.7152) + b*0.0722) / n                          (draw.fs lumaCoefs)
 *   var    = (m2/n - mean*mean) * (n / (n - 1))
 *   active = n < min_samples  ||  sqrt(max(var, 0) / n) > max_rel_error * max(mean, 1e-3)
 * A pixel that is not rendered keeps its sum, count and moment, so under a fixed threshold it never becomes active
 * again: the ticks a pixel received are always a prefix of the render's ticks, and it equals, bit for bit, the uniform
 * sum-mode render after that many ticks.  The moment m2 is a frame-sized f32 buffer, allocated (zeroed) when adaptive
 * sampling is first turned on and zeroed by fspt_clear; while adaptive sampling is on, every sample adds l*l, l =
 * (c.r*0.2126 + c.g*0.7152) + c.b*0.0722 of its colour after the NaN sanitising and the clamp (tracer.fs:515), in tick
 * order.  Renders with adaptive sampling off do not update it.
 * Counters: fspt_stats.samples counts the path samples actually rendered (counted on the device);
 * fspt_accum_device_ptr's n_samples stays the number of ticks; fspt_debug_last_color keeps the older value for the
 * pixels a wave did not render.
 * Multi-GPU: tile sharding composes (each rank decides for its own pixels; reduce and resolve are unchanged).
 * Sample-set sharding does not: one pixel's samples are split across ranks, and no rank sees its whole history. */
int fspt_set_adaptive(fspt_ctx* ctx, float max_rel_error, int32_t min_samples);
/* The number of pixels of the rectangle the next wave would render (the rule above on the current state); synchronises
 * the context's stream.  A host loop stops when it returns 0.  FSPT_E_STATE while adaptive sampling is off. */
int fspt_active_pixels(fspt_ctx* ctx, uint64_t* n_out);
/* The moment buffer, width*height f32 in GL order (next to fspt_read_accum / fspt_write_accum: a resumed adaptive render
 * writes back both).  FSPT_E_STATE before adaptive sampling has been turned on for the first time. */
int fspt_read_moment(fspt_ctx* ctx, float* out);
int fspt_write_moment(fspt_ctx* ctx, const float* in);

/* ---- multi-GPU: one context per GPU (one process per GPU, or several contexts in one process) ------------------
 * The reference renders one image on one GPU, one sample per requestAnimationFrame (main.js:838-857); every (pixel,
 * sample) of tracer.fs main() (:436-518) is independent, so the frame shards by image TILES and by SAMPLE SETS
 * (README.md:26-28 lists "Tiled rendering" as a TODO).  Collectives run inside the library on the context's stream
 * over NCCL (NVLink / NVSwitch); NCCL is dlopen'ed at fspt_comm_init, single-GPU hosts never load it. */

/* The pixel rectangle of the frame this context renders (gl.scissor-style, GL row order); default = whole frame.
 * camera.fs / tracer.fs see the same gl_FragCoord and resolution as in a whole-frame render, so a pixel's samples
 * are bit-identical whichever rectangle contains it.  The accumulation target stays frame-sized. */
int fspt_set_tile(fspt_ctx* ctx, int32_t x0, int32_t y0, int32_t width, int32_t height);

#define FSPT_COMM_ID_BYTES 128
/* ncclGetUniqueId: called once (by rank 0); the host ships the 128 bytes to the other ranks by any means. */
int fspt_comm_unique_id(uint8_t* id_out);
/* ncclCommInitRank on the context's device; collective over all `world` contexts. */
int fspt_comm_init(fspt_ctx* ctx, const uint8_t* id, int32_t rank, int32_t world);
int fspt_comm_destroy(fspt_ctx* ctx);
/* Sum of every rank's accumulation target -> root's, in place (ncclReduce, f32, 16 bytes/pixel), enqueued on the
 * context's stream after the renders already queued; sum mode only.  Collective. */
int fspt_reduce_accum(fspt_ctx* ctx, int32_t root);
/* The scene uploaded on `root` (fspt_scene_upload / _async) -> every other rank, device to device (ncclBroadcast of the
 * records the upload built + the environment and atlas texels): replaces the per-GPU repetition of the texImage
 * uploads of initBVH() (main.js:408-437,548-560).  Collective, in two phases: the geometry and the environment travel
 * at the call; the atlas part is issued by the rank's next fspt_render (behind its primary traversal launch, so an
 * asynchronous upload on the root overlaps on every rank), fspt_synchronize, fspt_reduce_accum, upload or broadcast,
 * whichever comes first -- like any collective, every rank has to reach one of them. */
int fspt_scene_broadcast(fspt_ctx* ctx, int32_t root);

/* mode=test (main.js:882-884, bvh_test.fs:224-232): one drawCamera() + primary intersectScene with the
 * visit counter.  Exports what bvh_test.fs computes but does not write out: result.index, result.t, count.
 * Also returns the camera targets (camera.fs:44-45) when pos4/dir4 are non-NULL (RGBA32F). */
int fspt_debug_primary(fspt_ctx* ctx, const fspt_frame_params* frame, float rand_base_camera,
                       int32_t* index_out, float* t_out, int32_t* count_out, float* pos4_out, float* dir4_out);

/* intersectScene (tracer.fs:366-404) on caller-supplied rays (RGBA32F pos/dir like the camera targets). */
int fspt_debug_trace(fspt_ctx* ctx, const float* pos4, const float* dir4, int32_t n_rays,
                     int32_t* index_out, float* t_out, int32_t* count_out);

/* Per-sample clamped colour of the LAST sample rendered (what tracer.fs computes before the running mean,
 * tracer.fs:515), RGBA32F; parity aid. */
int fspt_debug_last_color(fspt_ctx* ctx, float* rgba32f_out);

/* FSPT-DM2 arithmetic probes evaluated ON THE DEVICE (fn: 0 sin, 1 cos, 2 atan2(y,x), 3 asin, 4 exp2,
 * 5 pow(x,y)); parity aid for the platform built-ins the shaders rely on (tracer.fs:181,412,417). */
int fspt_debug_math(fspt_ctx* ctx, int32_t fn, const float* x, const float* y, float* out, int32_t n);

/* The host half of fspt_scene_upload without a GPU: pre-passes (interior-record numbering, material ids, depth / tree
 * check) and the device records the upload DMAs -- Node64 (n_interior x 16 floats), Tri48 ((n_triangles + 3) x 12), ShadeRec
 * (n_triangles x 48), the material id of every triangle.  info_out[5] = {n_interior, n_materials, root reference,
 * any dielectric, tree depth}.  Call with node64_out == NULL first to learn n_interior.  Test aid (the CPU suite checks the
 * records against the reference layout, main.js:360-392); errors are reported like fspt_scene_upload's, text through
 * fspt_last_error(NULL). */
int fspt_debug_pack_scene(const fspt_scene_desc* scene, float* node64_out, float* tri48_out, float* shaderec_out,
                          int32_t* mat_id_out, int32_t* info_out, int32_t n_threads);

/* Streaming-read microbenchmark on the context's device: `iters` passes over a `bytes`-sized buffer with L1-bypassing
 * 16-byte loads from a persistent grid; GB/s out.  With bytes well below the L2 size this is the L2->SM read
 * ceiling that bounds the traversal kernel (SURVEY 8d asks for this denominator); with bytes >> L2 it is the HBM
 * read ceiling.  Measurement aid, no reference counterpart. */
int fspt_debug_read_bandwidth(fspt_ctx* ctx, uint64_t bytes, int32_t iters, double* gb_per_s_out);

/* Tuning / behaviour switches (none changes an image).  Unknown keys return FSPT_E_INVALID. */
enum {
  FSPT_PARAM_ANYHIT = 1,          /* 1 (default): rays whose outcome is only tested for hit-or-miss -- every shadow ray
                                     (tracer.fs:501-502) and the continuation ray of a path's last bounce (:507-512 with
                                     i == NUM_BOUNCES-1) -- stop at their first intersection.  Same image bit for bit, fewer
                                     node visits than the reference's full traversal; 0 = full closest-hit traversal for
                                     every ray (the visit counters then equal the reference's). */
  FSPT_PARAM_MAX_REFRACTIONS = 2, /* safety cap of the unbounded refraction loop (tracer.fs:488), default 64 */
  FSPT_PARAM_SANITIZE_NAN = 3     /* default 1; no effect in practice: clamp() already maps NaN to 0 (DESIGN.md 2) */
};
int fspt_set_param(fspt_ctx* ctx, int32_t key, int32_t value);

int fspt_get_stats(fspt_ctx* ctx, fspt_stats* out);
int fspt_synchronize(fspt_ctx* ctx);

/* ---- host-side scene compilers that feed the path (rows f1, f3 of SURVEY.md section 8) ------------------ */

/* new BVH(triangles, maxTris) + serializeTree() + the flatten loop (bvh.js:5-50, main.js:355-392).
 * verts: n_tris*9 float64 world-space vertices (Triangle.verts).  nodes_out: capacity (2*n_tris)*9 f32,
 * receives the masked bvhBuffer; order_out[n_tris]: source triangle of every triTex slot (leaf order).
 * Bit-identical to the JavaScript builder; multi-threaded.  No GPU needed. */
int fspt_bvh_build(const double* verts, int32_t n_tris, int32_t max_tris, float* nodes_out, int32_t* order_out,
                   int32_t* n_nodes_out, int32_t* depth_out, int32_t n_threads);

/* Same, for scenes with `normalize` (main.js:337-348): box_verts = the vertices BEFORE the rescale, which is what
 * Triangle.boundingBox still holds (presorts + SAH sweeps), verts = the rescaled vertices (node boxes).  NULL = verts. */
int fspt_bvh_build2(const double* verts, const double* box_verts, int32_t n_tris, int32_t max_tris, float* nodes_out,
                    int32_t* order_out, int32_t* n_nodes_out, int32_t* depth_out, int32_t n_threads);

/* The same tree built on CUDA device `device` (sm_100 only): bit-identical to fspt_bvh_build2 on the same inputs, the same
 * outputs (nodes_out, order_out, n_nodes, depth) and the same refusals with the same codes (FSPT_E_INVALID for NaN / inf
 * vertices or bad arguments, FSPT_E_LIMIT where bvh.js would not terminate).  Synchronous: the call uploads the vertices,
 * builds, downloads the results, frees its device memory and stream and restores the caller's current device; it does
 * not synchronise the device, so a live context there keeps running.  Text of a failure through fspt_last_error(NULL).
 * Without a usable sm_100 device it fails with FSPT_E_CUDA (no CPU fallback). */
int fspt_bvh_build_device(int32_t device, const double* verts, const double* box_verts, int32_t n_tris, int32_t max_tris,
                          float* nodes_out, int32_t* order_out, int32_t* n_nodes_out, int32_t* depth_out);
/* FSPT_OK when `device` is a usable sm_100 device (what the device entry points need), FSPT_E_CUDA or FSPT_E_INVALID with
 * text through fspt_last_error(NULL) otherwise.  Lets a host choose between the two builders without trying one. */
int fspt_device_check(int32_t device);

/* ProcessEnvRadiance(img) (env_sampler.js:1-74) on an RGBA8 RGBE image; bins_out capacity in u16. */
int fspt_env_bins(const uint8_t* rgba8, int32_t width, int32_t height, uint16_t* bins_out, int32_t capacity,
                  int32_t* n_u16_out);

/* One image layer of TexturePacker.getPixels() (texture_packer.js:44-62): the WebGLTextureWriter blit
 * (:103-121,159-184) -- bilinear resample to res x res, y flip, sRGB decode when `corrected` (base-colour maps),
 * swizzle, premultiply by alpha, 8-bit quantise.  rgba8: w*h*4, row 0 = image top.  out: res*res*4, row 0 = GL row 0.
 * swizzle: 4 channel indices or NULL.  Host code, multi-threaded. */
int fspt_pack_layer(const uint8_t* rgba8, int32_t w, int32_t h, int32_t res, int32_t corrected, const int32_t* swizzle,
                    uint8_t* out, int32_t n_threads);

#ifdef __cplusplus
}
#endif
#endif /* FSPT_B200_H */
