/*
 * chunkycu.h - C ABI of libchunkycu.so, the B200-native (sm_100a CUDA) replacement for the OpenCL
 * device layer of the ChunkyCL plugin.
 *
 * This is the drop-in boundary: every entry point replaces a group of JOCL calls in the reference
 * (file:line citations are into /root/reference/src/main/java/dev/thatredox/chunkynative/).  A Java
 * host binds them through JNI or the FFM API (INTEGRATION.md shows the stubs); the Python host in
 * chunkyclplugin_b200/ binds the same symbols through ctypes.
 *
 * Conventions
 *   - plain C types only; host pointers are read/written during the call and never retained
 *     (the reference passes Pointer.to(javaArray) with blocking transfers, e.g. ClIntBuffer.java:22-24);
 *   - every function returns CCU_OK (0) or a negative CCU_E* code; ccu_last_error() returns the
 *     message of the calling thread's last failure (the reference runs with
 *     CL.setExceptionsEnabled(true), RendererInstance.java:36 - the Java shim turns non-zero into
 *     RuntimeException);
 *   - a ccu_ctx is bound to one CUDA device and is internally locked: entry points may be called from
 *     any thread (render thread, ForkJoin merge tasks, the cleaner thread - SURVEY.md 8b "threading");
 *   - there is no CPU fallback: without a CUDA device every call fails with CCU_ENODEVICE.
 */
#ifndef CHUNKYCU_H
#define CHUNKYCU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CCU_OK 0
#define CCU_ENODEVICE (-1) /* no CUDA device / driver (UnsatisfiedLinkError path, opencl/ChunkyCl.java:37-40) */
#define CCU_EINVAL (-2)    /* bad argument or call order */
#define CCU_ECUDA (-3)     /* a CUDA runtime call failed */
#define CCU_ENOMEM (-4)
#define CCU_ESTATE (-5)    /* scene/camera/render target not ready */

typedef struct ccu_ctx ccu_ctx;

/* launch parameters; the reference hard-codes 256 / 5 / 13.0f (rayTracer.cl:94,99,103,107) */
typedef struct ccu_render_params {
    int32_t draw_depth;    /* octree march step limit */
    int32_t max_depth;     /* ray depth limit (5 = 4 bounces) */
    float emitter_scale;   /* emitter intensity factor */
    int32_t kernel;        /* 0 = auto (4 when the commit-time layouts could be built, else 1), 1 = thread-per-pixel kernel (one launch per batch; cross-check and fallback), 4 = persistent wavefront kernel with a CTA-wide path pool and per-stage work masks */
    int32_t flags;         /* CCU_RENDER_* bits: Chunky's scene toggles as launch parameters (reference README.md:31-35) */
} ccu_render_params;
/* "Draw entities" unchecked: both entity BVHs are treated as empty (the reference gets EMPTY_NODE uploads from Chunky,
 * AbstractSceneLoader.java:118-127) without touching the uploaded scene. */
#define CCU_RENDER_NO_ENTITIES 1
/* Sunlight disabled (indoor scenes): bit 0 of the sun flags (PackedSun.java:16, tested at sky.h:45,69) reads as 0 - no sun
 * sampling, no sun disc - without re-uploading sunData. */
#define CCU_RENDER_NO_SUN 2
/* Specular, metallic and rough materials (beyond the reference, which shades every surface diffuse): word 5 of a material
 * (specular bits 0-7, metalness 8-15, roughness 16-23, each byte / 255) picks at every path-segment hit a metal event with
 * probability metalness, else a specular one with probability specular.  Such an event reflects the ray about the normal,
 * blended towards a diffuse direction by the roughness, takes no sun sample and tints the throughput by the surface colour
 * only for a metal.  A material whose word 5 is 0 shades as without the flag.  DESIGN.md "Beyond the reference: specular
 * materials" holds the exact contract. */
#define CCU_RENDER_SPECULAR 4
/* Emitter sampling (next-event estimation; beyond the reference, which finds a block emitter only when a diffuse bounce hits
 * it): at every diffuse path-segment hit whose bounce will be traced, one full-cube emitter voxel near the hit (the emitter
 * list of its grid cell) is sampled with a point on one of its faces facing the hit, and a shadow ray delivers its light;
 * the bounce then leaves out the emission of an emitter that list covered.  On flat-coloured emitters the image's
 * expectation is unchanged.  On textured ones (colour or emittance from the atlas) it is not exactly: the sample reads the
 * texel at the sampled point, while the reference's full-cube block test reads a texel shifted by its marched-position quirk
 * (SURVEY Q2), so the two weight the texture differently.  Quads, AABB models (see CCU_RENDER_EMITTER_MODELS) and triangles
 * keep the reference's behaviour.
 * A scene without full-cube emitters renders exactly as without the flag.  Both render kernels implement it.  DESIGN.md §10
 * holds the exact contract. */
#define CCU_RENDER_EMITTER_SAMPLING 8
/* Near-field emitter sampling, valid only together with CCU_RENDER_EMITTER_SAMPLING (ccu_render_set_params refuses it alone):
 * when the sampled emitter voxel lies within 1/8 of the hit (distance to its box), the sample is a cosine-weighted direction
 * scored when it enters the voxel, instead of a point on a face.  The area sampler's weight grows without bound as a hit
 * approaches an emitter face, which shows as fireflies where a surface meets an emitter; with this flag every sample's
 * contribution is bounded.  Farther emitters are sampled exactly as without it, and the image's expectation is that of
 * CCU_RENDER_EMITTER_SAMPLING.  DESIGN.md §11 holds the exact contract. */
#define CCU_RENDER_EMITTER_NEAR_FIELD 128
/* Model emitters, valid only together with CCU_RENDER_EMITTER_SAMPLING (ccu_render_set_params refuses it alone): emitter
 * sampling also samples quad models (torches, candles, end rods) and AABB models (lanterns, campfires) with an emitting quad or
 * box face, by a point on one of those primitives (with CCU_RENDER_EMITTER_NEAR_FIELD, by direction when the hit lies within
 * 1/8 of them), and the bounce leaves out their emission where the list covered them.  The image's expectation is that of
 * the flags without it, with the textured full-cube caveat above for full cubes only.  A scene without model emitters renders
 * exactly as with CCU_RENDER_EMITTER_SAMPLING alone.  Triangles keep the reference's behaviour.  DESIGN.md §12 holds the
 * exact contract. */
#define CCU_RENDER_EMITTER_MODELS 256
/* Biome tints (beyond the reference, which gives every grass, foliage and water surface one fixed colour): on a scene with biome
 * colours (ccu_scene_set_biome_colors), a material of tint type 1 (foliage), 2 (grass) or 3 (water) on a full cube, an AABB
 * model face or a quad of octree voxel (x, y, z) is tinted by the colour of its tint type at column (x, z) instead of the fixed
 * tint, where that column's chunk has colours; the alpha is multiplied by 255/256 as with the fixed tint.  Emitter samples
 * (CCU_RENDER_EMITTER_SAMPLING) read the colour at the emitter's voxel.  Triangles, tint 0xFF and chunks without colours keep the
 * reference's behaviour, and a scene without biome colours renders exactly as without the flag.  Valid alone and with every
 * other flag; both render kernels implement it.  DESIGN.md §13 holds the exact contract. */
#define CCU_RENDER_BIOME_TINT 512
/* Fog (beyond the reference; Chunky's uniform fog with sunlit light shafts): on a scene with fog (ccu_scene_set_fog, sigma > 0),
 * every path segment that hits is attenuated by exp(-sigma * length) and, with the sun on, gains one sun sample from a point
 * drawn uniformly along it, traced towards the sun without a limit; a segment that misses sees the sky blended towards the fog
 * colour by elevation.  Shadow and emitter-sample rays see neither.  A scene without fog renders exactly as without the flag.
 * Valid alone and with every other flag; both render kernels implement it.  DESIGN.md §14 holds the exact contract. */
#define CCU_RENDER_FOG 1024
/* Clouds (beyond the reference; Chunky's flat cloud layer): on a scene with a cloud layer (ccu_scene_set_clouds, a mask with a set
 * cell), every ray the render kernels trace also meets the cloud boxes: a path segment that enters one before its octree / BVH hit
 * hits a white diffuse surface that emits nothing, takes the sun sample and the diffuse bounce and no specular event or emitter
 * sample; sun shadow rays, emitter-sample rays and fog rays that meet a cloud are blocked, so clouds cast shadows.  A scene
 * without clouds renders exactly as without the flag.  First hit and preview do not see clouds.  Valid alone and with every
 * other flag; both render kernels implement it.  DESIGN.md §15 holds the exact contract. */
#define CCU_RENDER_CLOUDS 2048

/* ---- device enumeration: RendererInstance.java:39-75,123-157 (clGetPlatformIDs/clGetDeviceIDs/clGetDeviceInfo),
 *      used by the GPU selector UI (ui/GpuSelector.java:24-87) -------------------------------------------------- */
int ccu_device_count(int *count);
int ccu_device_info(int index, char *name, int name_len, int *sm_count, int *clock_khz, uint64_t *mem_bytes);

/* ---- context: RendererInstance.java:81-101 (clCreateContext + clCreateCommandQueue); no runtime compile step
 *      (KernelLoader.java:17-60 has no equivalent: kernels are built ahead of time for sm_100a) ----------------- */
int ccu_ctx_create(int device_index, ccu_ctx **out);
int ccu_ctx_destroy(ccu_ctx *ctx); /* idempotent on NULL; ClMemory.java:12-16 / NativeCleaner.java:38-53 */
const char *ccu_last_error(void);
const char *ccu_version(void);

/* ---- scene upload: ClSceneLoader.java:39-63, ClIntBuffer.java:14-25, ClPackedResourcePalette.java:14-26,
 *      AbstractSceneLoader.java:60-162.  Arrays use the reference's packed int layouts unchanged; zero-length
 *      arrays are accepted (the reference uploads a single 0 int, ClIntBuffer.java:15-18). ---------------------- */
int ccu_scene_begin(ccu_ctx *ctx);
int ccu_scene_set_octree(ccu_ctx *ctx, const int32_t *tree_data, int64_t n, int32_t depth); /* ClSceneLoader.java:52-63 (leaves already remapped, :56-58) */
int ccu_scene_set_block_palette(ccu_ctx *ctx, const int32_t *words, int64_t n);    /* ClSceneLoader.getBlockPalette :110 */
int ccu_scene_set_quad_models(ccu_ctx *ctx, const int32_t *words, int64_t n);      /* getQuadPalette :125 */
int ccu_scene_set_aabb_models(ccu_ctx *ctx, const int32_t *words, int64_t n);      /* getAabbPalette :120 */
int ccu_scene_set_material_palette(ccu_ctx *ctx, const int32_t *words, int64_t n); /* getMaterialPalette :115 */
int ccu_scene_set_triangles(ccu_ctx *ctx, const int32_t *words, int64_t n);        /* getTrigPalette :130 */
int ccu_scene_set_world_bvh(ccu_ctx *ctx, const int32_t *words, int64_t n);        /* getWorldBvh :135 */
int ccu_scene_set_actor_bvh(ccu_ctx *ctx, const int32_t *words, int64_t n);        /* getActorBvh :139 */
/* Biome colours for CCU_RENDER_BIOME_TINT (optional; beyond the reference).  chunks = n x {cx, cz}: chunk (cx, cz) covers voxels
 * 16 cx <= x < 16 cx + 16 and 16 cz <= z < 16 cz + 16 at every y; rgb = n x 3 planes x 256 texels x 3 floats, planes in tint-type
 * order (foliage, grass, water), texel (z & 15) * 16 + (x & 15), linear RGB as Chunky stores it.  CCU_EINVAL for n < 0, a null
 * array with n > 0, a negative coordinate, a duplicate chunk or a negative or non-finite component; n = 0 removes the colours.
 * ccu_scene_begin removes them too.  ccu_scene_commit fails with CCU_EINVAL when a chunk lies outside the octree's
 * max(1, 2^depth / 16) chunks per axis, or when the chunks' bounding box holds more than 2^24 chunks (the lookup grid covers
 * that box: every chunk of a depth-16 octree fits). */
int ccu_scene_set_biome_colors(ccu_ctx *ctx, const int32_t *chunks, const float *rgb, int64_t n);
/* Fog for CCU_RENDER_FOG (optional; beyond the reference).  sigma = extinction per block (>= 0, finite; 0 removes the fog),
 * sky_density = Chunky's sky fog density in [0, 1], color = linear RGB fog colour (3 floats, each >= 0 and finite), fast = Chunky's
 * "fast fog" switch (0 or 1).  CCU_EINVAL otherwise.  Like the sun it belongs to the scene: ccu_scene_begin removes it, and it
 * takes effect at the next ccu_scene_commit (ccu_group_replicate_scene carries it). */
int ccu_scene_set_fog(ccu_ctx *ctx, float sigma, float sky_density, const float color[3], int32_t fast);
/* Cloud layer for CCU_RENDER_CLOUDS (optional; beyond the reference).  mask = 256 x 256 bytes, non-zero = cloud; cell (i, k) is
 * mask[(k & 255) * 256 + (i & 255)].  A point (x, y, z) of the plugin's frame (world minus scene origin, as for camera rays) is in a
 * cloud when y0 <= y <= y1 and cell (floor(x / size + u0), floor(z / size + v0)) is set (1 / size is computed once, in fp32).
 * CCU_EINVAL for a size that is not positive and finite, a y0, y1, u0 or v0 that is not finite, or y0 >= y1; mask = NULL removes
 * the clouds (the other arguments are then ignored).  Like the fog it belongs to the scene: ccu_scene_begin removes it, and it
 * takes effect at the next ccu_scene_commit (ccu_group_replicate_scene carries it).  The committed scene holds the mask
 * bit-packed (8 KiB, counted by ccu_scene_device_bytes). */
int ccu_scene_set_clouds(ccu_ctx *ctx, const uint8_t *mask, float size, float y0, float y1, float u0, float v0);
/* texture atlas: ClTextureLoader.java:46-66 - clCreateImage(8192x8192xlayers RGBA8) then one clEnqueueWriteImage
 * per texture at (16*tileX, 16*tileY, layer) */
int ccu_scene_atlas_create(ccu_ctx *ctx, int32_t width, int32_t height, int32_t layers);
int ccu_scene_atlas_write(ccu_ctx *ctx, int32_t x, int32_t y, int32_t layer, int32_t w, int32_t h, const uint8_t *rgba);
/* whole-image convenience (row-major [layers][height][width][4]) */
int ccu_scene_set_atlas(ccu_ctx *ctx, const uint8_t *rgba, int32_t width, int32_t height, int32_t layers);
int ccu_scene_set_sky(ccu_ctx *ctx, const uint8_t *rgba, int32_t resolution, float sky_intensity); /* ClSky.java:23-62 */
int ccu_scene_set_sun(ccu_ctx *ctx, const int32_t sun_words[6]);                                   /* ClSceneLoader.getSun :148, PackedSun.java:31-41 */
int ccu_scene_commit(ccu_ctx *ctx); /* builds the traversal layout in HBM; scene is immutable until the next begin */

/* ---- camera: ClCamera.java:33-70 (settings buffer) and :72-105 (pre-generated ray upload) -------------------- */
int ccu_camera_set(ccu_ctx *ctx, int32_t projector_type, const float *settings, int64_t n_floats);

/* ---- path tracing: OpenClPathTracingRenderer.java:54-191 ------------------------------------------------------ */
int ccu_render_begin(ccu_ctx *ctx, int32_t width, int32_t height);   /* :71-78 accumulation buffer (zeros), width/height buffers */
int ccu_render_set_params(ccu_ctx *ctx, const ccu_render_params *p); /* optional; defaults = reference constants */
/* :102-144 for n_passes consecutive passes: pass i uses seeds[i] (the host draws rand.nextInt() per pass, :106-107)
 * and bufferSpp = passes already in the window (:108-109); blocks until the device is done (:141). */
int ccu_render_passes(ccu_ctx *ctx, const int32_t *seeds, int32_t n_passes);
int ccu_render_passes_async(ccu_ctx *ctx, const int32_t *seeds, int32_t n_passes); /* same, returns after enqueue */
int ccu_render_sync(ccu_ctx *ctx);
/* :164-166 blocking read of the running-mean buffer float[3*W*H]; *window_spp = passes accumulated in the window */
int ccu_render_read(ccu_ctx *ctx, float *mean_rgb, int32_t *window_spp);
/* :167-173 fused read + merge into Chunky's double sample buffer:
 *   sample[i] = (sample[i]*sample_spp + mean[i]*window_spp) / (sample_spp + window_spp); then the window restarts (:170) */
int ccu_render_merge(ccu_ctx *ctx, double *sample_buffer, int32_t sample_spp, int32_t *merged_spp);
/* :150-151,172-177 the reference merges in a ForkJoin task while the next passes render.  ccu_render_merge_async does the same:
 * it closes the window (the next passes go to a second accumulation buffer), starts the read-back on a copy stream and the
 * spp-weighted merge on worker threads, and returns.  `sample_buffer` must stay valid until ccu_render_merge_wait (or the next
 * merge / ccu_render_end, which wait implicitly).  *merged_spp = passes of the closed window. */
int ccu_render_merge_async(ccu_ctx *ctx, double *sample_buffer, int32_t sample_spp, int32_t *merged_spp);
int ccu_render_merge_wait(ccu_ctx *ctx);   /* bufferMergeTask.join() */
/* The same in two calls, for hosts that run the merge on a thread of their own (the Java shim: Chunky.getCommonThreads(), with the
 * heap array passed as a critical segment): ccu_render_window_close closes the window and starts the read-back (returns at once;
 * call it on the render thread before the next ccu_render_passes); ccu_render_window_merge - any thread - waits for the copies
 * and merges.  Exactly one merge per close. */
int ccu_render_window_close(ccu_ctx *ctx, int32_t *window_spp);
int ccu_render_window_merge(ccu_ctx *ctx, double *sample_buffer, int32_t sample_spp);
int ccu_render_reset_window(ccu_ctx *ctx); /* bufferSppReal = 0 (:170); the buffer itself is not cleared, as in the reference */
/* multi-GPU: after the window buffers of all ranks have been reduced into this context's buffer (mean over all passes), tell it how
 * many passes the buffer now stands for, so that ccu_render_merge / ccu_render_read weight it correctly (bufferSppReal of :167-173) */
int ccu_render_set_window_spp(ccu_ctx *ctx, int32_t window_spp);
int ccu_render_end(ccu_ctx *ctx);          /* releases the per-render buffers (:80-85 try-with-resources) */

/* multi-GPU plumbing: device pointer of the running-mean buffer (float[3*W*H]) so that the host's
 * communication layer (NCCL) can reduce per-GPU buffers without a host round trip, and a scaling hook
 * that turns the mean into a window sum (mean * window_spp) before the reduce. */
int ccu_render_device_buffer(ccu_ctx *ctx, void **device_ptr, int64_t *n_floats);
int ccu_render_scale(ccu_ctx *ctx, float factor);
int ccu_stream_handle(ccu_ctx *ctx, void **cuda_stream);

/* ---- first-hit buffers for the camera rays (BASELINE config 2); built on closestIntersect kernel.h:14-24 ------
 * block  = record.material (block palette pointer, 0 on miss)   face = 0..5 (-x,+x,-y,+y,-z,+z) or 6
 * node   = index of the hit leaf in the uploaded treeData (-1 on miss / BVH hit)
 * kind   = 0 miss, 1 octree, 2 world BVH, 3 actor BVH            t = record.distance (+inf on miss)
 * normal = float[3*W*H], color = float[4*W*H]; any output pointer may be NULL. */
int ccu_first_hit(ccu_ctx *ctx, int32_t seed, int32_t *block, int32_t *face, int32_t *node, int32_t *kind, float *t,
                  float *normal, float *color);

/* ---- preview: OpenClPreviewRenderer.java:47-115 (kernel rayTracer.cl:115-217), ARGB int[W*H] ----------------- */
int ccu_preview(ccu_ctx *ctx, int32_t *argb);

/* ---- post-processing filters: GpuPostProcessingFilter.processFrame (tonemap/GpuPostProcessingFilter.java:40-65), kernel
 *      tonemap/include/post_processing_filter.cl:5-51.  input = Chunky's double sample buffer (3 per pixel), argb = int[W*H];
 *      type: 0 GAMMA, 1 TONEMAP1, 2 ACES ("TONEMAP2"), 3 HABLE ("TONEMAP3") (ImposterCombinationGpuPostProcessingFilter.java:11-16) */
int ccu_tonemap(ccu_ctx *ctx, int32_t width, int32_t height, float exposure, const double *input, int32_t type, int32_t *argb);

/* ---- instrumentation ------------------------------------------------------------------------------------------ */
int ccu_last_kernel_ms(ccu_ctx *ctx, float *ms);          /* CUDA-event time of the last render_passes / first_hit launch(es) */
int ccu_launch_count(ccu_ctx *ctx, int64_t *launches);    /* kernels launched by this context so far */
/* Test support: the render kernel instance of the context's last ccu_render_passes[_async] launch (all zero before the first).
 * out = {kernel launched (1 or 4, after the choice for kernel 0), HAS_BVH, LAY (kernel 4) or MODE (kernel 1), spec, nee (a NeeKind:
 * 0 none, 1 area, 2 near, 3 area + models, 4 near + models), biome, sky texels staged in shared memory (0 for kernel 1)};
 * LAY is the one the launch ran (a fog launch may move from LAY 0 to LAY 1, DESIGN.md §5).
 * DESIGN.md §5.  A launch refused with an error leaves it as it was. */
int ccu_debug_last_render(ccu_ctx *ctx, int32_t out[7]);
/* The same report with the switches added since: writes the first min(n, 9) of {the 7 entries above, fog, clouds}. */
int ccu_debug_last_render_n(ccu_ctx *ctx, int32_t *out, int32_t n);
int ccu_scene_device_bytes(ccu_ctx *ctx, int64_t *bytes); /* HBM held by the committed scene */
int ccu_scene_commit_ms(ccu_ctx *ctx, double *ms);        /* host time the last ccu_scene_commit spent building + uploading the layouts */
/* Memory-system denominators for this path's roofline (dependent 32-byte-sector gathers, SURVEY 8d): random 16-byte
 * L2 loads over an array of `array_bytes` (4 MB = L2 resident, 1 GB = HBM resident); dependent = 1 walks a pointer chain
 * (ns_per_load = latency of one dependent gather), 0 issues independent loads (gbytes_per_s = sector bandwidth). */
int ccu_bench_gather(ccu_ctx *ctx, int64_t array_bytes, int32_t dependent, float *gbytes_per_s, float *ns_per_load);
/* Host-only (no CUDA call): what the two commit-time traversal layouts built from `tree` answer for `count` voxels
 * (xyz = count x 3 ints): the value-carrying layout's leaf value / level (-1 / -1 when a leaf value cannot be encoded)
 * and the march ("air") layout's not-air flag / air-leaf level (-1 when not air).  Both must agree with the reference's
 * root descent (octree.h:81-88, ClSceneLoader.java:56-59 numbering); used by the CPU test-suite. */
int ccu_debug_layout_lookup(const int32_t *tree, int64_t n, int32_t depth, const int32_t *xyz, int64_t count, int32_t *wide_value,
                            int32_t *wide_level, int32_t *air_solid, int32_t *air_level);

/* Test support, host only: the BVH stage layout ccu_scene_commit builds from a BinaryBVH.packed node array (bvh.h:47-110: 7 ints
 * per node {child / -leaf pointer, 6 box floats}) and the triangle palette (count + n x 20 ints per leaf, PackedTriangle.java:46-78).
 * rec: 16 words per inner node = two halves {box (6), ref, 0} of the first / second child; tris: per leaf {count, 0 x 7} +
 * count x 24 words, 8 words of zero padding at the end; ref >= 0 = inner record, ref < 0 = -(1 + leaf block offset / 8 words).
 * rec / tris may be NULL (sizes only); *ok = 0 when the node array cannot be laid out (malformed, or deeper than the 64 entries of
 * the reference's traversal stack, bvh.h:38).  Used by the CPU test-suite. */
int ccu_debug_bvh_layout(const int32_t *bvh, int64_t n_bvh, const int32_t *trigs, int64_t n_trigs, int32_t *rec, int64_t rec_cap,
                         int32_t *tris, int64_t tris_cap, int64_t *rec_words, int64_t *tris_words, int32_t *root, int32_t *ok);

/* Test support, host only: the emitter table of CCU_RENDER_EMITTER_SAMPLING that ccu_scene_commit builds from the reference's
 * octree node array and the block / material palettes (DESIGN.md §10).  info = {has_emitters, grid origin x y z (voxels), grid
 * size x y z (cells), log2 of the cell edge, emitters, list words}; emit (4 ints per emitter: x, y, z, block palette position,
 * sorted by x, y, z), off (cells + 1 offsets into list) and list may be NULL (sizes only) and must otherwise hold those sizes.
 * Used by the CPU test-suite. */
int ccu_debug_emitter_grid(const int32_t *tree, int64_t n_tree, int32_t depth, const int32_t *block_palette, int64_t n_block,
                           const int32_t *mat_palette, int64_t n_mat, int32_t info[10], int32_t *emit, int32_t *off, int32_t *list);
/* Test support, host only: the wider emitter table of CCU_RENDER_EMITTER_MODELS (DESIGN.md §12) that ccu_scene_commit builds
 * from the octree node array and the block / material / quad / AABB palettes.  info = {has_model_emitters, grid origin x y z,
 * grid size x y z, log2 of the cell edge, emitters, list words, head entries, primitive words}; emit, off and list as in
 * ccu_debug_emitter_grid; head (one int per block palette position: the int4 index of its primitive list in prim, -1 for no
 * model emitter) and prim (the headers {m, bounding box as 6 float bits, 0} and the 16-word primitive records) may be NULL
 * (sizes only) and must otherwise hold those sizes.  Used by the CPU test-suite. */
int ccu_debug_emitter_models(const int32_t *tree, int64_t n_tree, int32_t depth, const int32_t *block_palette, int64_t n_block,
                             const int32_t *mat_palette, int64_t n_mat, const int32_t *quad_models, int64_t n_quad,
                             const int32_t *aabb_models, int64_t n_aabb, int32_t info[12], int32_t *emit, int32_t *off,
                             int32_t *list, int32_t *head, int32_t *prim);

/* Test support, host only: the biome layout ccu_scene_commit builds from ccu_scene_set_biome_colors' arrays for an octree of
 * `depth` (DESIGN.md §13), with the same checks.  info = {x0, z0, gx, gz, tiles}: the grid covers the chunks' bounding box, gx x gz
 * chunks from chunk (x0, z0); grid (gx x gz ints, index (cx - x0) * gz + (cz - z0), the tile of the chunk or -1) and tiles (tiles
 * x 3 planes x 256 texels x 4 floats {r, g, b, 0}) may be NULL (sizes only) and must otherwise hold those sizes.  Used by the CPU
 * test-suite. */
int ccu_debug_biome_layout(const int32_t *chunks, const float *rgb, int64_t n, int32_t depth, int32_t info[5], int32_t *grid, float *tiles);

/* ---- multi-GPU: samples-per-pixel split over the GPUs of one box (SURVEY.md 8e) -------------------------------------------
 * The reference is one JVM and one device (RendererInstance.java:81-101).  A group is N contexts, each holding a full scene
 * replica; pass p of a window goes to member p mod N with the seed it would have had on one GPU (state = seed_p + gid,
 * rayTracer.cl:55), so the union of samples equals the 1-GPU run.  The only exchange is the sum of the per-GPU window buffers:
 * an NCCL reduce-scatter over NVLink, after which EVERY GPU copies its 1/N share to the host over its own PCIe link and the
 * shares are merged into the sample buffer in parallel (OpenClPathTracingRenderer.java:164-173 with passSpp = all passes).
 *
 * Two ways to form a group:
 *   ccu_group_create      one process drives all GPUs (the JVM plugin): ncclCommInitAll + one worker thread per device;
 *   ccu_group_join        one process per GPU (torchrun): every rank wraps its own context; rank 0 obtains an id with
 *                         ccu_group_unique_id and the host distributes it (any channel) before the collective join.
 * Scene: upload + commit on member 0 as usual, then ccu_group_replicate_scene copies the committed scene (layouts included)
 * to the other members device-to-device; with ccu_group_join every rank uploads its own replica. */
typedef struct ccu_group ccu_group;
#define CCU_UNIQUE_ID_BYTES 128
int ccu_group_create(const int32_t *devices, int32_t n, ccu_group **out);
int ccu_group_unique_id(uint8_t id[CCU_UNIQUE_ID_BYTES]);
int ccu_group_join(ccu_ctx *ctx, const uint8_t id[CCU_UNIQUE_ID_BYTES], int32_t rank, int32_t world, ccu_group **out);
int ccu_group_destroy(ccu_group *g);
int ccu_group_size(ccu_group *g, int32_t *world, int32_t *local_members);
int ccu_group_member(ccu_group *g, int32_t local_index, ccu_ctx **ctx);   /* borrowed; owned by the group for ccu_group_create */
int ccu_group_replicate_scene(ccu_group *g);                              /* member 0 -> all local members, over NVLink */
int ccu_group_camera_set(ccu_group *g, int32_t projector_type, const float *settings, int64_t n_floats);
int ccu_group_render_begin(ccu_group *g, int32_t width, int32_t height);
int ccu_group_render_set_params(ccu_group *g, const ccu_render_params *p);
/* seeds of ALL passes of the batch in 1-GPU order; member of global rank r renders passes r, r+N, ... (asynchronously) */
int ccu_group_render_passes(ccu_group *g, const int32_t *seeds, int32_t n_passes);
int ccu_group_render_sync(ccu_group *g);
/* reduce-scatter of the window sums, per-GPU read-back of its share, merge into sample_buffer (all shares with ccu_group_create;
 * only this rank's share - sample_buffer must then be memory shared by all ranks - with ccu_group_join).  Collective. */
int ccu_group_render_merge(ccu_group *g, double *sample_buffer, int32_t sample_spp, int32_t *merged_spp);
/* the same, returning once the reduce-scatter and the share read-backs are queued: the next window renders while the shares travel
 * and are merged (sample_buffer stays in use until ccu_group_render_merge_wait / the next merge / ccu_group_render_end). */
int ccu_group_render_merge_async(ccu_group *g, double *sample_buffer, int32_t sample_spp, int32_t *merged_spp);
int ccu_group_render_merge_wait(ccu_group *g);
/* only the device part of the merge: reduce-scatter of the open window (closes it; the sums stay on the GPUs until the next
 * ccu_group_render_merge reads them back).  *window_spp = passes of the window.  Collective. */
int ccu_group_render_reduce(ccu_group *g, int32_t *window_spp);
int ccu_group_render_end(ccu_group *g);
int ccu_group_last_ms(ccu_group *g, float *render_ms, float *reduce_ms);   /* device time of the last batch (max over local members) / last reduce-scatter */

#ifdef __cplusplus
}
#endif
#endif /* CHUNKYCU_H */
