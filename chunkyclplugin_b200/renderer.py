"""Host-side mirror of the reference's renderer classes, driving the C ABI instead of JOCL.

The reference's host is Java inside Chunky (no JVM or chunky-core in this image), so this module is the
host that stands in for it: same class roles, method names, call order and error behaviour as

  reference (dev.thatredox.chunkynative.opencl)        here
  -------------------------------------------------    -------------------------------------------
  renderer/RendererInstance.java                       RendererInstance
  renderer/ClSceneLoader.java (+ AbstractSceneLoader)  CudaSceneLoader   (alias ClSceneLoader)
  renderer/scene/ClCamera.java                         CudaCamera        (alias ClCamera)
  OpenClPathTracingRenderer.java                       CudaPathTracingRenderer (alias OpenClPathTracingRenderer)
  OpenClPreviewRenderer.java                           CudaPreviewRenderer     (alias OpenClPreviewRenderer)

``Scene`` / ``DefaultRenderManager`` are minimal stand-ins for the Chunky objects those classes touch
(sample buffer, spp counters, snapshot control, redraw).  The Java shim in java/ makes the same calls.
"""
from __future__ import annotations

import threading
import time
from typing import Callable, Optional

import numpy as np

from . import native
from .javarandom import JavaRandom
from .scenes import PackedScene


# ----------------------------------------------------------------------------------------------------
# Chunky stand-ins
# ----------------------------------------------------------------------------------------------------
class Scene:
    """What the renderers use of se.llbit.chunky.renderer.scene.Scene."""

    def __init__(self, packed: PackedScene, target_spp: int = 16, ray_generator: Optional[Callable[[bool], np.ndarray]] = None):
        self.packed = packed
        # projectorType -1 only: stands in for Camera.calcViewRay over all pixels (ClCamera.java:75-97); called with
        # jitter on/off, returns float32[6*W*H].  Without it the rays stored in the packed scene are used as they are.
        self.ray_generator = ray_generator
        self.width, self.height = packed.width, packed.height
        self.sample_buffer = np.zeros(self.width * self.height * 3, dtype=np.float64)   # getSampleBuffer()
        self.back_buffer = np.zeros(self.width * self.height, dtype=np.int32)           # getBackBuffer().data
        self.spp = 0
        self.target_spp = target_spp
        self.finalize_buffer = False
        self.post_process_calls = 0

    def getSampleBuffer(self): return self.sample_buffer
    def getTargetSpp(self): return self.target_spp
    def shouldFinalizeBuffer(self): return self.finalize_buffer
    def postProcessFrame(self): self.post_process_calls += 1


class SnapshotControl:
    """Save events: at the target spp and optionally every ``dump_frequency`` spp."""

    def __init__(self, dump_frequency: int = 0):
        self.dump_frequency = dump_frequency

    def saveSnapshot(self, scene: Scene, spp: int) -> bool:
        return spp >= scene.target_spp

    def saveRenderDump(self, scene: Scene, spp: int) -> bool:
        return self.dump_frequency > 0 and spp % self.dump_frequency == 0


class DefaultRenderManager:
    def __init__(self, scene: Scene, snapshot_control: Optional[SnapshotControl] = None):
        self.bufferedScene = scene
        self.snapshot_control = snapshot_control or SnapshotControl()
        self.redraws = 0

    def getSnapshotControl(self): return self.snapshot_control
    def redrawScreen(self): self.redraws += 1
    def shouldFinalize(self): return False


# ----------------------------------------------------------------------------------------------------
# RendererInstance.java:23-28,31-110 - device selection + context singleton
# ----------------------------------------------------------------------------------------------------
class RendererInstance:
    _instance: Optional["RendererInstance"] = None
    _lock = threading.Lock()
    persistent_settings = {"clDevice": 0}          # PersistentSettings int "clDevice" (RendererInstance.java:33)

    def __init__(self, device_index: Optional[int] = None):
        n = native.device_count()                   # raises (no fallback) when no CUDA device exists
        self.devices = [native.device_info(i) for i in range(n)]
        idx = self.persistent_settings.get("clDevice", 0) if device_index is None else device_index
        if not 0 <= idx < n:
            idx = 0                                 # RendererInstance.java:74: falls back to the first device
        self.device_index = idx
        self.context = native.Context(idx)

    @classmethod
    def get(cls, device_index: Optional[int] = None) -> "RendererInstance":
        with cls._lock:
            if cls._instance is None or (device_index is not None and cls._instance.device_index != device_index):
                if cls._instance is not None:
                    cls._instance.context.close()
                cls._instance = RendererInstance(device_index)
            return cls._instance

    @classmethod
    def reset(cls):
        with cls._lock:
            if cls._instance is not None:
                cls._instance.context.close()
            cls._instance = None


# ----------------------------------------------------------------------------------------------------
# ClSceneLoader.java + AbstractSceneLoader.java:42-162
# ----------------------------------------------------------------------------------------------------
def upload_scene(ctx, p) -> None:
    """Upload and commit a PackedScene through the C ABI in the order of the reference's loader (AbstractSceneLoader.java:60-162),
    with its biome colours, fog and clouds when it has them."""
    ctx.scene_begin()
    ctx.set_atlas(p.atlas)                      # ClTextureLoader.buildTextures
    ctx.set_block_palette(p.block_palette)
    ctx.set_material_palette(p.mat_palette)
    ctx.set_aabb_models(p.aabb_models)
    ctx.set_quad_models(p.quad_models)
    ctx.set_triangles(p.bvh_trigs)
    ctx.set_world_bvh(p.world_bvh)
    ctx.set_actor_bvh(p.actor_bvh)
    ctx.set_sun(p.sun)
    ctx.set_sky(p.sky, p.sky_intensity)         # ClSky
    if p.biome is not None:
        ctx.set_biome_colors(*p.biome)          # CCU_RENDER_BIOME_TINT's colours (beyond the reference)
    if p.fog is not None:
        ctx.set_fog(*p.fog)                     # CCU_RENDER_FOG's fog (beyond the reference)
    if p.clouds is not None:
        ctx.set_clouds(*p.clouds)               # CCU_RENDER_CLOUDS's cloud layer (beyond the reference)
    ctx.set_octree(p.octree, p.octree_depth)    # loadOctree, ClSceneLoader.java:52-63
    ctx.scene_commit()


class CudaSceneLoader:
    def __init__(self, instance: Optional[RendererInstance] = None):
        self.instance = instance or RendererInstance.get()
        self.modCount = 0
        self._loaded_scene_id = None

    def ensureLoad(self, scene: Scene) -> bool:                        # AbstractSceneLoader.java:42-55
        if self._loaded_scene_id != id(scene.packed):
            self.modCount = -1
            return self.load(0, "SCENE_LOADED", scene)
        return True

    def load(self, modCount: int, resetReason: str, scene: Scene) -> bool:    # :60-162
        if self.modCount == modCount:
            return True
        if resetReason in ("NONE", "MODE_CHANGE"):
            self.modCount = modCount
            return True
        upload_scene(self.instance.context, scene.packed)
        self.modCount = modCount
        self._loaded_scene_id = id(scene.packed)
        return True


# ----------------------------------------------------------------------------------------------------
# ClCamera.java:33-105
# ----------------------------------------------------------------------------------------------------
class CudaCamera:
    def __init__(self, scene: Scene, instance: Optional[RendererInstance] = None):
        self.instance = instance or RendererInstance.get()
        self.scene = scene
        self.projectorType = scene.packed.projector_type
        self.needGenerate = self.projectorType == -1
        if not self.needGenerate:
            self.instance.context.camera_set(self.projectorType, scene.packed.camera[:15])

    def generate(self, renderLock=None, jitter: bool = True):          # :72-105
        if not self.needGenerate:
            return
        gen = getattr(self.scene, "ray_generator", None)
        # fresh sub-pixel jitter per call (ThreadLocalRandom in the reference, :83-87); the packed rays are the jitter-free set
        rays = gen(jitter) if gen is not None else self.scene.packed.camera
        # The reference takes renderLock around the upload because its queue is shared with the pass loop (:99-104).  Here the
        # library uploads into the ray buffer no launch is reading, on its copy stream, so the upload overlaps the passes in
        # flight and the next ccu_render_passes picks the new rays up; the lock is not needed.
        self.instance.context.camera_set(-1, rays)
        self.generations = getattr(self, "generations", 0) + 1

    def close(self): pass


# ----------------------------------------------------------------------------------------------------
# OpenClPathTracingRenderer.java
# ----------------------------------------------------------------------------------------------------
class CudaPathTracingRenderer:
    MERGE_WINDOW = 1024                                       # :158
    CALLBACK_MS = 100.0                                       # :153-157 postRender is polled at most every 100 ms

    def __init__(self, sceneLoader: Optional[CudaSceneLoader] = None, passes_per_call: int = 0, merge_window: Optional[int] = None,
                 camera_regen_passes: int = 8):
        self.sceneLoader = sceneLoader or CudaSceneLoader()
        self.postRender: Callable[[], bool] = lambda: False   # Chunky passes a callback that returns true to stop
        # How many passes one C-ABI call may cover.  The reference issues 1 per launch and polls postRender at most every
        # 100 ms; here a call covers as many passes as fit in about CALLBACK_MS of device time (measured, so heavy scenes get
        # short batches and the UI stays responsive), never more than up to the next merge point.  > 0 pins the batch size.
        self.passes_per_call = passes_per_call
        self.merge_window = merge_window or self.MERGE_WINDOW
        # projectorType -1: passes rendered with one set of camera rays before a freshly jittered set may replace it
        self.camera_regen_passes = max(1, camera_regen_passes)
        self.kernel_ms = 0.0
        self._ms_per_pass: Optional[float] = None             # device time per pass of the last batch (kept across renders)

    def getId(self): return "ChunkyClRenderer"               # :33-36 - the renderer selector id is unchanged
    def getName(self): return "ChunkyClRenderer"
    def getDescription(self): return "ChunkyClRenderer"
    def setPostRender(self, callback): self.postRender = callback
    def autoPostProcess(self): return False                  # :197-200

    def sceneReset(self, manager: DefaultRenderManager, reason: str, resetCount: int):     # :203-205
        self.sceneLoader.load(resetCount, reason, manager.bufferedScene)

    def _batch_limit(self) -> int:
        if self.passes_per_call > 0:
            return self.passes_per_call
        if self._ms_per_pass is None:
            return 1                                         # first call: one pass, to learn what a pass costs
        return max(1, int(self.CALLBACK_MS / max(self._ms_per_pass, 1e-3)))

    def render(self, manager: DefaultRenderManager):         # :54-191
        instance = self.sceneLoader.instance
        ctx = instance.context
        renderLock = threading.Lock()
        scene = manager.bufferedScene
        sampleBuffer = scene.getSampleBuffer()

        self.sceneLoader.ensureLoad(scene)                   # :64
        camera = CudaCamera(scene, instance)                 # :70
        ctx.render_begin(scene.width, scene.height)          # :71-78
        cameraGenTask: Optional[threading.Thread] = None
        cameraErrors = []
        mergePending = [False]

        def finishMerge():                                   # bufferMergeTask.join() + the tail of the merge task (:174-176)
            if mergePending[0]:
                ctx.render_merge_wait()
                mergePending[0] = False
                scene.postProcessFrame()
                manager.redrawScreen()

        def cameraGen():
            try:
                camera.generate(renderLock, True)
            except Exception as e:                           # surfaced on the render thread
                cameraErrors.append(e)

        try:
            camera.generate(renderLock, True)                # :88
            bufferSppReal = 0
            logicalSpp = scene.spp
            sceneSpp = scene.spp
            rand = JavaRandom(0)                             # :95
            self.kernel_ms = 0.0
            lastCallback = 0.0
            while logicalSpp < scene.getTargetSpp():         # :102
                # The reference issues one pass per launch and tests for a save event after each (:150).  Here one
                # C-ABI call covers all passes up to the next point where the reference would merge - the next save
                # event (snapshot / dump / target spp) or a full window, found by probing the same predicate - but no
                # more than the batch limit (about 100 ms of device time, or camera_regen_passes with generated rays).
                n = max(1, min(self.merge_window - bufferSppReal, self._batch_limit()))
                if camera.needGenerate:
                    n = min(n, self.camera_regen_passes)
                control = manager.getSnapshotControl()
                for k in range(1, n + 1):
                    if self._isSaveEvent(control, scene, logicalSpp + bufferSppReal + k):
                        n = k
                        break
                seeds = np.array([rand.next_int() for _ in range(n)], dtype=np.int32)      # :106-107
                with renderLock:
                    ctx.render_passes(seeds)                 # :108-141 (bufferSpp tracked by the library)
                ms = ctx.last_kernel_ms()
                self.kernel_ms += ms
                self._ms_per_pass = ms / n
                bufferSppReal += n                           # :143-144
                scene.spp += n
                if cameraErrors:
                    raise cameraErrors[0]
                if camera.needGenerate and (cameraGenTask is None or not cameraGenTask.is_alive()):    # :146-148
                    cameraGenTask = threading.Thread(target=cameraGen, daemon=True)
                    cameraGenTask.start()
                saveEvent = self._isSaveEvent(manager.getSnapshotControl(), scene, logicalSpp + bufferSppReal)
                if not scene.shouldFinalizeBuffer() and not saveEvent:
                    now = time.monotonic() * 1e3
                    if now - lastCallback > self.CALLBACK_MS and not manager.shouldFinalize():    # :153-157
                        lastCallback = now
                        if self.postRender():
                            break
                    if bufferSppReal < self.merge_window:    # :158-159
                        continue
                finishMerge()                                # :162 bufferMergeTask.join()
                if self.postRender():                        # :163
                    break
                # :164-173 read + weighted merge + window reset; like the reference's ForkJoin task the merge runs in the
                # background (copy stream + worker threads of the library) while the next passes render
                passSpp = ctx.render_merge_async(sampleBuffer, sceneSpp)
                mergePending[0] = True
                assert passSpp == bufferSppReal
                sceneSpp += passSpp
                bufferSppReal = 0
                logicalSpp += passSpp                        # :178
                if saveEvent:                                # :179-182
                    finishMerge()
                    if self.postRender():
                        break
        finally:
            if cameraGenTask is not None:
                cameraGenTask.join()                         # :186
            try:
                finishMerge()                                # :187
            finally:
                camera.close()
                ctx.render_end()
        if cameraErrors:
            raise cameraErrors[0]

    def render_features(self, manager: DefaultRenderManager, spp: int):
        """The denoiser's feature buffers of the buffered scene (DESIGN.md §16): (albedo, normal), Chunky-layout float64[3*W*H]
        each, the first-hit means over `spp` passes whose seeds are drawn as render() draws them (JavaRandom(0), one nextInt per
        pass).  With a projector the library generates the rays, so these are the camera rays of the first `spp` passes of
        render().  With pre-generated rays (projector -1) one freshly jittered ray set serves every pass, whereas render()
        switches to a new set every `camera_regen_passes` passes (whenever the background upload lands), so the jitter differs
        from render()'s.  A render of more than CCU_FEATURES_MAX_PASSES passes is split into calls of at most that many, whose
        means are combined in double."""
        if spp < 1:
            raise ValueError("render_features needs at least one pass")
        ctx = self.sceneLoader.instance.context
        scene = manager.bufferedScene
        self.sceneLoader.ensureLoad(scene)
        camera = CudaCamera(scene, self.sceneLoader.instance)
        ctx.render_begin(scene.width, scene.height)
        try:
            camera.generate(None, True)
            rand = JavaRandom(0)
            seeds = np.array([rand.next_int() for _ in range(spp)], dtype=np.int32)
            albedo = normal = None
            done = 0
            for off in range(0, spp, native.CCU_FEATURES_MAX_PASSES):
                part = seeds[off:off + native.CCU_FEATURES_MAX_PASSES]
                a, n = ctx.render_features(part)
                if albedo is None:
                    albedo, normal = a.astype(np.float64), n.astype(np.float64)
                else:
                    albedo = (albedo * done + a.astype(np.float64) * part.size) / (done + part.size)
                    normal = (normal * done + n.astype(np.float64) * part.size) / (done + part.size)
                done += part.size
        finally:
            camera.close()
            ctx.render_end()
        return albedo, normal

    def denoise(self, manager: DefaultRenderManager, feature_spp: int = 16, iterations: int = 5,
                sigma_luminance: float = 4.0) -> np.ndarray:
        """The buffered scene's sample buffer denoised on the GPU (DESIGN.md §17): render_features(manager, feature_spp), then
        the guided a-trous filter of the sample buffer with those albedo and normal buffers.  Returns a new Chunky-layout
        float64[3*W*H], ready for GpuPostProcessingFilter.processFrame or pfm.write_pfm; the sample buffer stays as it was."""
        scene = manager.bufferedScene
        albedo, normal = self.render_features(manager, feature_spp)
        ctx = self.sceneLoader.instance.context
        return ctx.denoise(scene.sample_buffer, albedo.astype(np.float32), normal.astype(np.float32), iterations,
                           sigma_luminance, width=scene.width, height=scene.height)

    @staticmethod
    def _isSaveEvent(control: SnapshotControl, scene: Scene, spp: int) -> bool:           # :193-195
        return control.saveSnapshot(scene, spp) or control.saveRenderDump(scene, spp)


# ----------------------------------------------------------------------------------------------------
# OpenClPreviewRenderer.java:47-115
# ----------------------------------------------------------------------------------------------------
class CudaPreviewRenderer:
    def __init__(self, sceneLoader: Optional[CudaSceneLoader] = None):
        self.sceneLoader = sceneLoader or CudaSceneLoader()

    def getId(self): return "ChunkyClPreviewRenderer"
    def getName(self): return "ChunkyClPreviewRenderer"
    def getDescription(self): return "ChunkyClPreviewRenderer"
    def autoPostProcess(self): return False

    def sceneReset(self, manager, reason, resetCount):
        self.sceneLoader.load(resetCount, reason, manager.bufferedScene)

    def render(self, manager: DefaultRenderManager):
        scene = manager.bufferedScene
        ctx = self.sceneLoader.instance.context
        self.sceneLoader.ensureLoad(scene)
        camera = CudaCamera(scene, self.sceneLoader.instance)
        ctx.render_begin(scene.width, scene.height)
        try:
            camera.generate(None, False)
            scene.back_buffer[:] = ctx.preview()
            manager.redrawScreen()
        finally:
            ctx.render_end()


# ----------------------------------------------------------------------------------------------------
# tonemap/GpuPostProcessingFilter.java, ImposterCombinationGpuPostProcessingFilter.java, ChunkyCl.java:59-71
# ----------------------------------------------------------------------------------------------------
class BitmapImage:
    """Stand-in for se.llbit.chunky.resources.BitmapImage: ARGB ints, row-major."""

    def __init__(self, width: int, height: int):
        self.width, self.height = width, height
        self.data = np.zeros(width * height, dtype=np.int32)


class GpuPostProcessingFilter:
    """PostProcessingFilter that shadows one of Chunky's filters (same name / id) with the device kernel."""

    class Filter:                                             # ImposterCombinationGpuPostProcessingFilter.java:11-16
        GAMMA, TONEMAP1, ACES, HABLE = 0, 1, 2, 3

    # ChunkyCl.java:59-62: which Chunky filter id each kernel type shadows
    IMPOSTERS = {"GAMMA": Filter.GAMMA, "TONEMAP1": Filter.TONEMAP1, "TONEMAP2": Filter.ACES, "TONEMAP3": Filter.HABLE}

    def __init__(self, filter_id: str, instance: Optional[RendererInstance] = None, name: Optional[str] = None,
                 description: Optional[str] = None):
        if filter_id not in self.IMPOSTERS:
            raise KeyError(f"no device filter shadows {filter_id!r}")
        self.id, self.filter = filter_id, self.IMPOSTERS[filter_id]
        self.name = name or filter_id
        self.description = description or filter_id
        self.instance = instance or RendererInstance.get()

    def getName(self): return self.name
    def getDescription(self): return self.description
    def getId(self): return self.id

    def processFrame(self, width: int, height: int, input: np.ndarray, output: BitmapImage, exposure: float, task=None):   # :40-65
        output.data[:] = self.instance.context.tonemap(width, height, float(exposure), input, self.filter)


# reference-named aliases, so code written against the reference's class names reads the same
ClSceneLoader = CudaSceneLoader
ClCamera = CudaCamera
OpenClPathTracingRenderer = CudaPathTracingRenderer
OpenClPreviewRenderer = CudaPreviewRenderer
