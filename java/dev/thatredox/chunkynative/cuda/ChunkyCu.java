package dev.thatredox.chunkynative.cuda;

import java.lang.foreign.*;
import java.lang.invoke.MethodHandle;

import static java.lang.foreign.ValueLayout.*;

/**
 * Java FFM (JDK 22+, java.lang.foreign; critical downcalls with heap segments need 22) binding of libchunkycu.so - include/chunkycu.h.
 *
 * Drop-in replacement for the JOCL calls of the reference plugin; one method per C entry point.  A JNI variant
 * is a mechanical translation (see INTEGRATION.md).  NOT COMPILED in the build image (no JDK there).
 *
 * Every call returns the C status; {@link #check(int)} turns a non-zero status into a RuntimeException carrying
 * ccu_last_error(), which preserves the reference's behaviour under CL.setExceptionsEnabled(true)
 * (RendererInstance.java:36).  A missing library surfaces as UnsatisfiedLinkError / IllegalArgumentException from
 * SymbolLookup, which ChunkyCl.attach already catches to disable the plugin (ChunkyCl.java:37-40).
 */
public final class ChunkyCu {
    private static final Linker LINKER = Linker.nativeLinker();
    private static final SymbolLookup LIB = SymbolLookup.libraryLookup(System.mapLibraryName("chunkycu"), Arena.global());

    private static MethodHandle h(String name, FunctionDescriptor fd) {
        return LINKER.downcallHandle(LIB.find(name).orElseThrow(() -> new UnsatisfiedLinkError(name)), fd);
    }

    private static final MethodHandle DEVICE_COUNT = h("ccu_device_count", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle DEVICE_INFO = h("ccu_device_info", FunctionDescriptor.of(JAVA_INT, JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, ADDRESS));
    private static final MethodHandle CTX_CREATE = h("ccu_ctx_create", FunctionDescriptor.of(JAVA_INT, JAVA_INT, ADDRESS));
    private static final MethodHandle CTX_DESTROY = h("ccu_ctx_destroy", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle LAST_ERROR = h("ccu_last_error", FunctionDescriptor.of(ADDRESS));
    private static final MethodHandle SCENE_BEGIN = h("ccu_scene_begin", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle SET_OCTREE = h("ccu_scene_set_octree", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_INT));
    private static final FunctionDescriptor WORDS = FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG);
    private static final MethodHandle SET_BLOCKS = h("ccu_scene_set_block_palette", WORDS);
    private static final MethodHandle SET_QUADS = h("ccu_scene_set_quad_models", WORDS);
    private static final MethodHandle SET_AABBS = h("ccu_scene_set_aabb_models", WORDS);
    private static final MethodHandle SET_MATERIALS = h("ccu_scene_set_material_palette", WORDS);
    private static final MethodHandle SET_TRIANGLES = h("ccu_scene_set_triangles", WORDS);
    private static final MethodHandle SET_WORLD_BVH = h("ccu_scene_set_world_bvh", WORDS);
    private static final MethodHandle SET_ACTOR_BVH = h("ccu_scene_set_actor_bvh", WORDS);
    private static final MethodHandle SET_BIOME_COLORS = h("ccu_scene_set_biome_colors", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG));
    private static final MethodHandle SET_FOG = h("ccu_scene_set_fog", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_FLOAT, JAVA_FLOAT, ADDRESS, JAVA_INT));
    private static final MethodHandle SET_CLOUDS = h("ccu_scene_set_clouds", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_FLOAT, JAVA_FLOAT, JAVA_FLOAT, JAVA_FLOAT, JAVA_FLOAT));
    private static final MethodHandle DEBUG_BIOME_LAYOUT = h("ccu_debug_biome_layout", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_INT, ADDRESS, ADDRESS, ADDRESS));
    private static final MethodHandle ATLAS_CREATE = h("ccu_scene_atlas_create", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT));
    private static final MethodHandle ATLAS_WRITE = h("ccu_scene_atlas_write", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, ADDRESS));
    private static final MethodHandle SET_SKY = h("ccu_scene_set_sky", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, JAVA_FLOAT));
    private static final MethodHandle SET_SUN = h("ccu_scene_set_sun", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    private static final MethodHandle SCENE_COMMIT = h("ccu_scene_commit", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle CAMERA_SET = h("ccu_camera_set", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, JAVA_LONG));
    private static final MethodHandle RENDER_BEGIN = h("ccu_render_begin", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT));
    private static final MethodHandle RENDER_SET_PARAMS = h("ccu_render_set_params", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    private static final MethodHandle RENDER_PASSES = h("ccu_render_passes", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT));
    private static final MethodHandle RENDER_PASSES_ASYNC = h("ccu_render_passes_async", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT));
    private static final MethodHandle RENDER_SYNC = h("ccu_render_sync", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle WINDOW_CLOSE = h("ccu_render_window_close", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    // the merge reads and writes Chunky's double[] in place: a critical downcall may take the heap array itself (no 50 MB copy)
    private static final MethodHandle WINDOW_MERGE = LINKER.downcallHandle(LIB.find("ccu_render_window_merge").orElseThrow(() -> new UnsatisfiedLinkError("ccu_render_window_merge")),
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT), Linker.Option.critical(true));
    private static final MethodHandle LAST_KERNEL_MS = h("ccu_last_kernel_ms", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    private static final MethodHandle RENDER_READ = h("ccu_render_read", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS));
    private static final MethodHandle RENDER_MERGE = LINKER.downcallHandle(LIB.find("ccu_render_merge").orElseThrow(() -> new UnsatisfiedLinkError("ccu_render_merge")),
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS), Linker.Option.critical(true));
    private static final MethodHandle RENDER_END = h("ccu_render_end", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle PREVIEW = h("ccu_preview", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    private static final MethodHandle RENDER_FEATURES = h("ccu_render_features", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, ADDRESS));
    private static final MethodHandle TONEMAP = h("ccu_tonemap", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, JAVA_FLOAT, ADDRESS, JAVA_INT, ADDRESS));
    private static final MethodHandle DENOISE = h("ccu_denoise", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_INT, JAVA_FLOAT, ADDRESS));
    // multi-GPU group (include/chunkycu.h "multi-GPU"): one JVM drives all GPUs of the box
    private static final MethodHandle GROUP_CREATE = h("ccu_group_create", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, ADDRESS));
    private static final MethodHandle GROUP_DESTROY = h("ccu_group_destroy", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle GROUP_MEMBER = h("ccu_group_member", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, ADDRESS));
    private static final MethodHandle GROUP_REPLICATE = h("ccu_group_replicate_scene", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle GROUP_CAMERA_SET = h("ccu_group_camera_set", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, JAVA_LONG));
    private static final MethodHandle GROUP_RENDER_BEGIN = h("ccu_group_render_begin", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT));
    private static final MethodHandle GROUP_RENDER_SET_PARAMS = h("ccu_group_render_set_params", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    private static final MethodHandle GROUP_RENDER_PASSES = h("ccu_group_render_passes", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT));
    private static final MethodHandle GROUP_RENDER_SYNC = h("ccu_group_render_sync", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle GROUP_RENDER_MERGE = LINKER.downcallHandle(LIB.find("ccu_group_render_merge").orElseThrow(() -> new UnsatisfiedLinkError("ccu_group_render_merge")),
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS), Linker.Option.critical(true));
    private static final MethodHandle GROUP_RENDER_END = h("ccu_group_render_end", FunctionDescriptor.of(JAVA_INT, ADDRESS));

    /** ccu_render_params.flags: Chunky's "draw entities" / sunlight toggles as launch parameters (reference README.md:31-35), and
     *  specular / metallic / rough materials from material word 5 (beyond the reference, DESIGN "Beyond the reference: specular materials"). */
    public static final int RENDER_NO_ENTITIES = 1, RENDER_NO_SUN = 2, RENDER_SPECULAR = 4, RENDER_EMITTER_SAMPLING = 8;
    /** ccu_render_params.flags: near-field emitter sampling (DESIGN §11), valid only together with RENDER_EMITTER_SAMPLING. */
    public static final int RENDER_EMITTER_NEAR_FIELD = 128;
    /** ccu_render_params.flags: emitter sampling also samples quad and AABB model emitters (DESIGN §12), valid only together
     *  with RENDER_EMITTER_SAMPLING. */
    public static final int RENDER_EMITTER_MODELS = 256;
    /** ccu_render_params.flags: grass, foliage and water tinted by the biome colours of {@link Context#setBiomeColors} (DESIGN §13). */
    public static final int RENDER_BIOME_TINT = 512;
    /** ccu_render_params.flags: the scene's fog of {@link Context#setFog}, with sunlit light shafts (DESIGN §14). */
    public static final int RENDER_FOG = 1024;
    /** ccu_render_params.flags: the scene's cloud layer of {@link Context#setClouds}, which also shadows the scene (DESIGN §15). */
    public static final int RENDER_CLOUDS = 2048;
    private static final StructLayout RENDER_PARAMS = MemoryLayout.structLayout(JAVA_INT.withName("draw_depth"), JAVA_INT.withName("max_depth"),
            JAVA_FLOAT.withName("emitter_scale"), JAVA_INT.withName("kernel"), JAVA_INT.withName("flags"));

    private ChunkyCu() {}

    static void check(int rc) {
        if (rc != 0) {
            String msg;
            try {
                msg = ((MemorySegment) LAST_ERROR.invokeExact()).reinterpret(512).getString(0);
            } catch (Throwable t) {
                msg = "?";
            }
            throw new RuntimeException("chunkycu error " + rc + ": " + msg);
        }
    }

    /** Floats per chunk of ccu_scene_set_biome_colors' rgb array: 3 planes x 256 texels x 3. */
    private static final int BIOME_TILE_FLOATS = 3 * 256 * 3;

    /** The arrays must hold the n chunks they are passed for: 2n ints and 2304n floats (the native side reads that many). */
    static void checkBiomeArrays(int[] chunks, float[] rgb, int n) {
        if (n < 0 || (n > 0 && (chunks == null || rgb == null || chunks.length < 2L * n || rgb.length < (long) BIOME_TILE_FLOATS * n)))
            throw new IllegalArgumentException("biome colours: arrays too short for " + n + " chunks");
    }

    /** Test support: the biome layout commit builds for an octree of {@code depth}; returns {x0, z0, gx, gz, tiles} and fills grid
     *  (gx * gz ints) and tiles (tiles * 3 * 256 * 4 floats) when they are large enough (include/chunkycu.h,
     *  ccu_debug_biome_layout). */
    public static int[] debugBiomeLayout(int[] chunks, float[] rgb, int n, int depth, int[] grid, float[] tiles) {
        checkBiomeArrays(chunks, rgb, n);
        try (Arena a = Arena.ofConfined()) {
            MemorySegment c = n > 0 ? a.allocateFrom(JAVA_INT, java.util.Arrays.copyOf(chunks, 2 * n)) : MemorySegment.NULL;
            MemorySegment r = n > 0 ? a.allocateFrom(JAVA_FLOAT, java.util.Arrays.copyOf(rgb, BIOME_TILE_FLOATS * n)) : MemorySegment.NULL;
            MemorySegment info = a.allocate(JAVA_INT, 5);
            check((int) DEBUG_BIOME_LAYOUT.invokeExact(c, r, (long) n, depth, info, MemorySegment.NULL, MemorySegment.NULL));
            int[] out = info.toArray(JAVA_INT);
            long cells = (long) out[2] * out[3], floats = (long) out[4] * 3 * 256 * 4;
            if (grid != null && tiles != null && grid.length >= cells && tiles.length >= floats) {
                MemorySegment gs = a.allocate(JAVA_INT, Math.max(cells, 1)), ts = a.allocate(JAVA_FLOAT, Math.max(floats, 1));
                check((int) DEBUG_BIOME_LAYOUT.invokeExact(c, r, (long) n, depth, info, gs, ts));
                MemorySegment.copy(gs, JAVA_INT, 0, grid, 0, (int) cells);
                MemorySegment.copy(ts, JAVA_FLOAT, 0, tiles, 0, (int) floats);
            }
            return out;
        } catch (RuntimeException e) {
            throw e;
        } catch (Throwable t) {
            throw new RuntimeException(t);
        }
    }

    /** One ccu_ctx; AutoCloseable like the reference's ClMemory handles (ClMemory.java:12-29). */
    public static final class Context implements AutoCloseable {
        private MemorySegment handle;
        private final boolean owned;

        /** A member context of a {@link Group}: borrowed, closed with the group. */
        Context(MemorySegment borrowed) { handle = borrowed; owned = false; }

        public Context(int deviceIndex) {
            owned = true;
            try (Arena a = Arena.ofConfined()) {
                MemorySegment out = a.allocate(ADDRESS);
                check((int) CTX_CREATE.invokeExact(deviceIndex, out));
                handle = out.get(ADDRESS, 0);
            } catch (RuntimeException e) {
                throw e;
            } catch (Throwable t) {
                throw new RuntimeException(t);
            }
        }

        private static int call(MethodHandle mh, Object... args) {
            try {
                return (int) mh.invokeWithArguments(args);
            } catch (Throwable t) {
                throw new RuntimeException(t);
            }
        }

        private void words(MethodHandle mh, int[] data, int length) {
            try (Arena a = Arena.ofConfined()) {
                MemorySegment seg = a.allocateFrom(JAVA_INT, java.util.Arrays.copyOf(data, Math.max(length, 0)));
                check(call(mh, handle, seg, (long) length));
            }
        }

        public void sceneBegin() { check(call(SCENE_BEGIN, handle)); }
        /** ClSceneLoader.loadOctree: leaves already remapped to block palette pointers (ClSceneLoader.java:56-58). */
        public void setOctree(int[] treeData, int depth) {
            try (Arena a = Arena.ofConfined()) {
                check(call(SET_OCTREE, handle, a.allocateFrom(JAVA_INT, treeData), (long) treeData.length, depth));
            }
        }
        public void setBlockPalette(int[] w, int n) { words(SET_BLOCKS, w, n); }
        public void setQuadModels(int[] w, int n) { words(SET_QUADS, w, n); }
        public void setAabbModels(int[] w, int n) { words(SET_AABBS, w, n); }
        public void setMaterialPalette(int[] w, int n) { words(SET_MATERIALS, w, n); }
        public void setTriangles(int[] w, int n) { words(SET_TRIANGLES, w, n); }
        public void setWorldBvh(int[] w) { words(SET_WORLD_BVH, w, w.length); }
        public void setActorBvh(int[] w) { words(SET_ACTOR_BVH, w, w.length); }
        /** Biome colours of n chunks: chunks = n x {cx, cz}, rgb = n x 3 planes (foliage, grass, water) x 256 texels x 3 linear floats,
         *  texel (z &amp; 15) * 16 + (x &amp; 15).  n = 0 removes them. */
        public void setBiomeColors(int[] chunks, float[] rgb, int n) {
            checkBiomeArrays(chunks, rgb, n);
            try (Arena a = Arena.ofConfined()) {
                MemorySegment c = n > 0 ? a.allocateFrom(JAVA_INT, java.util.Arrays.copyOf(chunks, 2 * n)) : MemorySegment.NULL;
                MemorySegment r = n > 0 ? a.allocateFrom(JAVA_FLOAT, java.util.Arrays.copyOf(rgb, BIOME_TILE_FLOATS * n)) : MemorySegment.NULL;
                check(call(SET_BIOME_COLORS, handle, c, r, (long) n));
            }
        }
        /** The scene's fog: extinction per block (0 removes it), Chunky's sky fog density in [0, 1], a linear RGB colour, fast fog. */
        public void setFog(float sigma, float skyDensity, float[] color, boolean fast) {
            if (color.length != 3) throw new IllegalArgumentException("the fog colour needs 3 components");
            try (Arena a = Arena.ofConfined()) {
                check(call(SET_FOG, handle, sigma, skyDensity, a.allocateFrom(JAVA_FLOAT, color), fast ? 1 : 0));
            }
        }
        /** The scene's cloud layer: mask = 256 x 256 bytes (cell (i, k) at (k &amp; 255) * 256 + (i &amp; 255), non-zero = cloud; null removes
         *  the layer), cell size, the slab y0 &lt; y1 and the cell offsets u0, v0, in the plugin's frame (DESIGN §15). */
        public void setClouds(byte[] mask, float size, float y0, float y1, float u0, float v0) {
            if (mask != null && mask.length != 256 * 256) throw new IllegalArgumentException("the cloud mask needs 256 x 256 cells");
            try (Arena a = Arena.ofConfined()) {
                MemorySegment m = mask != null ? a.allocateFrom(JAVA_BYTE, mask) : MemorySegment.NULL;
                check(call(SET_CLOUDS, handle, m, size, y0, y1, u0, v0));
            }
        }
        public void atlasCreate(int width, int height, int layers) { check(call(ATLAS_CREATE, handle, width, height, layers)); }
        /** One call per texture, as clEnqueueWriteImage in ClTextureLoader.java:60-66. */
        public void atlasWrite(int x, int y, int layer, int w, int h, byte[] rgba) {
            try (Arena a = Arena.ofConfined()) {
                check(call(ATLAS_WRITE, handle, x, y, layer, w, h, a.allocateFrom(JAVA_BYTE, rgba)));
            }
        }
        public void setSky(byte[] rgba, int resolution, float intensity) {
            try (Arena a = Arena.ofConfined()) {
                check(call(SET_SKY, handle, a.allocateFrom(JAVA_BYTE, rgba), resolution, intensity));
            }
        }
        public void setSun(int[] sunWords) {
            try (Arena a = Arena.ofConfined()) {
                check(call(SET_SUN, handle, a.allocateFrom(JAVA_INT, sunWords)));
            }
        }
        public void sceneCommit() { check(call(SCENE_COMMIT, handle)); }
        public void cameraSet(int projectorType, float[] settings) {
            try (Arena a = Arena.ofConfined()) {
                check(call(CAMERA_SET, handle, projectorType, a.allocateFrom(JAVA_FLOAT, settings), (long) settings.length));
            }
        }
        public void renderBegin(int width, int height) { check(call(RENDER_BEGIN, handle, width, height)); }
        /** drawDepth (scene ray depth UI), maxDepth, emitter scale, kernel (0 = auto) and the RENDER_* toggles. */
        public void renderSetParams(int drawDepth, int maxDepth, float emitterScale, int kernel, int flags) {
            try (Arena a = Arena.ofConfined()) {
                MemorySegment p = a.allocate(RENDER_PARAMS);
                p.set(JAVA_INT, 0, drawDepth); p.set(JAVA_INT, 4, maxDepth); p.set(JAVA_FLOAT, 8, emitterScale);
                p.set(JAVA_INT, 12, kernel); p.set(JAVA_INT, 16, flags);
                check(call(RENDER_SET_PARAMS, handle, p));
            }
        }
        public void renderPasses(int[] seeds) {
            try (Arena a = Arena.ofConfined()) {
                check(call(RENDER_PASSES, handle, a.allocateFrom(JAVA_INT, seeds), seeds.length));
            }
        }
        /** Returns after the enqueue; renderSync() waits (without holding the context lock, so previews / tonemaps go through). */
        public void renderPassesAsync(int[] seeds) {
            try (Arena a = Arena.ofConfined()) {
                check(call(RENDER_PASSES_ASYNC, handle, a.allocateFrom(JAVA_INT, seeds), seeds.length));
            }
        }
        public void renderSync() { check(call(RENDER_SYNC, handle)); }
        public float lastKernelMs() {
            try (Arena a = Arena.ofConfined()) {
                MemorySegment ms = a.allocate(JAVA_FLOAT);
                check(call(LAST_KERNEL_MS, handle, ms));
                return ms.get(JAVA_FLOAT, 0);
            }
        }
        /** Fused read + weighted merge into Chunky's sample buffer (OpenClPathTracingRenderer.java:164-173); blocking. */
        public int renderMerge(double[] sampleBuffer, int sampleSpp) {
            try (Arena a = Arena.ofConfined()) {
                MemorySegment merged = a.allocate(JAVA_INT);
                check(call(RENDER_MERGE, handle, MemorySegment.ofArray(sampleBuffer), sampleSpp, merged));
                return merged.get(JAVA_INT, 0);
            }
        }
        /** Closes the window (the next passes go to the second buffer) and starts its read-back; returns its pass count. */
        public int windowClose() {
            try (Arena a = Arena.ofConfined()) {
                MemorySegment n = a.allocate(JAVA_INT);
                check(call(WINDOW_CLOSE, handle, n));
                return n.get(JAVA_INT, 0);
            }
        }
        /** The merge of the closed window; runs on a Chunky common-pool thread while the render thread queues the next passes. */
        public void windowMerge(double[] sampleBuffer, int sampleSpp) {
            check(call(WINDOW_MERGE, handle, MemorySegment.ofArray(sampleBuffer), sampleSpp));
        }
        public void renderEnd() { check(call(RENDER_END, handle)); }
        public void preview(int[] argb) {
            try (Arena a = Arena.ofConfined()) {
                MemorySegment out = a.allocate(JAVA_INT, argb.length);
                check(call(PREVIEW, handle, out));
                MemorySegment.copy(out, JAVA_INT, 0, argb, 0, argb.length);
            }
        }

        /** The denoiser's feature buffers (DESIGN §16): the first-hit albedo and normal averaged over the passes with these seeds,
         *  3 floats per pixel each; either array may be null, not both (include/chunkycu.h, ccu_render_features). */
        public void renderFeatures(int[] seeds, float[] albedo, float[] normal) {
            try (Arena a = Arena.ofConfined()) {
                MemorySegment s = a.allocateFrom(JAVA_INT, seeds);
                MemorySegment al = albedo != null ? a.allocate(JAVA_FLOAT, albedo.length) : MemorySegment.NULL;
                MemorySegment no = normal != null ? a.allocate(JAVA_FLOAT, normal.length) : MemorySegment.NULL;
                check((int) RENDER_FEATURES.invokeExact(handle, s, seeds.length, al, no));
                if (albedo != null) MemorySegment.copy(al, JAVA_FLOAT, 0, albedo, 0, albedo.length);
                if (normal != null) MemorySegment.copy(no, JAVA_FLOAT, 0, normal, 0, normal.length);
            }
        }

        /** GpuPostProcessingFilter.processFrame (tonemap/GpuPostProcessingFilter.java:40-65): filter = Filter.id (0..3). */
        public void tonemap(int width, int height, double[] input, int[] argb, double exposure, int filter) {
            try (Arena a = Arena.ofConfined()) {
                MemorySegment in = a.allocateFrom(JAVA_DOUBLE, input);
                MemorySegment out = a.allocate(JAVA_INT, argb.length);
                check(call(TONEMAP, handle, width, height, (float) exposure, in, filter, out));
                MemorySegment.copy(out, JAVA_INT, 0, argb, 0, argb.length);
            }
        }

        /** The guided a-trous denoiser (DESIGN §17): color = the double[3*W*H] sample buffer, albedo and normal = the float
         *  feature buffers of renderFeatures, out = double[3*W*H] (may be color itself); defaults iterations 5,
         *  sigmaLuminance 4 (include/chunkycu.h, ccu_denoise). */
        public void denoise(int width, int height, double[] color, float[] albedo, float[] normal, int iterations,
                            float sigmaLuminance, double[] out) {
            try (Arena a = Arena.ofConfined()) {
                MemorySegment c = a.allocateFrom(JAVA_DOUBLE, color);
                MemorySegment al = a.allocateFrom(JAVA_FLOAT, albedo);
                MemorySegment no = a.allocateFrom(JAVA_FLOAT, normal);
                MemorySegment o = a.allocate(JAVA_DOUBLE, out.length);
                check(call(DENOISE, handle, width, height, c, al, no, iterations, sigmaLuminance, o));
                MemorySegment.copy(o, JAVA_DOUBLE, 0, out, 0, out.length);
            }
        }

        @Override
        public void close() {
            if (handle != null) {
                if (owned) call(CTX_DESTROY, handle);
                handle = null;
            }
        }
    }

    /** N GPUs rendering one image (ccu_group_*): scene uploaded to member 0 and replicated over NVLink, passes striped, one
     *  NCCL reduce-scatter per window, every GPU merging its share of the sample buffer. */
    public static final class Group implements AutoCloseable {
        private MemorySegment handle;
        public final int size;

        public Group(int[] devices) {
            try (Arena a = Arena.ofConfined()) {
                MemorySegment out = a.allocate(ADDRESS);
                check((int) GROUP_CREATE.invokeExact(a.allocateFrom(JAVA_INT, devices), devices.length, out));
                handle = out.get(ADDRESS, 0);
                size = devices.length;
            } catch (RuntimeException e) {
                throw e;
            } catch (Throwable t) {
                throw new RuntimeException(t);
            }
        }
        /** Member 0 is the context the scene loader uploads to. */
        public Context member(int i) {
            try (Arena a = Arena.ofConfined()) {
                MemorySegment out = a.allocate(ADDRESS);
                check(Context.call(GROUP_MEMBER, handle, i, out));
                return new Context(out.get(ADDRESS, 0));
            }
        }
        public void replicateScene() { check(Context.call(GROUP_REPLICATE, handle)); }
        public void cameraSet(int projectorType, float[] settings) {
            try (Arena a = Arena.ofConfined()) {
                check(Context.call(GROUP_CAMERA_SET, handle, projectorType, a.allocateFrom(JAVA_FLOAT, settings), (long) settings.length));
            }
        }
        public void renderBegin(int width, int height) { check(Context.call(GROUP_RENDER_BEGIN, handle, width, height)); }
        public void renderPasses(int[] seeds) {
            try (Arena a = Arena.ofConfined()) {
                check(Context.call(GROUP_RENDER_PASSES, handle, a.allocateFrom(JAVA_INT, seeds), seeds.length));
            }
        }
        public void renderSync() { check(Context.call(GROUP_RENDER_SYNC, handle)); }
        public int renderMerge(double[] sampleBuffer, int sampleSpp) {
            try (Arena a = Arena.ofConfined()) {
                MemorySegment merged = a.allocate(JAVA_INT);
                check(Context.call(GROUP_RENDER_MERGE, handle, MemorySegment.ofArray(sampleBuffer), sampleSpp, merged));
                return merged.get(JAVA_INT, 0);
            }
        }
        public void renderEnd() { check(Context.call(GROUP_RENDER_END, handle)); }
        @Override public void close() {
            if (handle != null) { Context.call(GROUP_DESTROY, handle); handle = null; }
        }
    }

    /** Device name for the GPU selector (ui/GpuSelector.java:89-125 reads CL_DEVICE_NAME). */
    public static String deviceName(int index) {
        try (Arena a = Arena.ofConfined()) {
            MemorySegment name = a.allocate(256);
            check((int) DEVICE_INFO.invokeExact(index, name, 256, MemorySegment.NULL, MemorySegment.NULL, MemorySegment.NULL));
            return name.getString(0);
        } catch (RuntimeException e) {
            throw e;
        } catch (Throwable t) {
            throw new RuntimeException(t);
        }
    }

    public static int deviceCount() {
        try (Arena a = Arena.ofConfined()) {
            MemorySegment n = a.allocate(JAVA_INT);
            check((int) DEVICE_COUNT.invokeExact(n));
            return n.get(JAVA_INT, 0);
        } catch (RuntimeException e) {
            throw e;
        } catch (Throwable t) {
            throw new RuntimeException(t);
        }
    }
}
