"""Round-2 features of the C ABI on the GPU: scene toggles as launch parameters, scene re-use on one context, deep worlds,
deep BVHs, overlapped merge and camera-ray uploads.  All against the CPU oracle, bit-exact."""
import dataclasses
import threading

import numpy as np
import pytest

from chunkyclplugin_b200.javarandom import pass_seeds
from conftest import load_scene
from oracle.edge_rays import embed_octree

pytestmark = pytest.mark.gpu


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _render(ctx, seeds):
    ctx.render_passes(np.asarray(seeds, np.int32))
    return ctx.render_read()[0]


# ---------------------------------------------------------------------------------------------------------
# Chunky's scene toggles (reference README.md:31-35) as launch parameters
# ---------------------------------------------------------------------------------------------------------
def test_draw_entities_off_is_the_scene_without_bvhs(scenes, cuda_ctx):
    """CCU_RENDER_NO_ENTITIES == what Chunky uploads with "draw entities" unchecked: EMPTY_NODE BVHs (AbstractSceneLoader.java:118-127)."""
    import oracle
    from chunkyclplugin_b200 import native
    from chunkyclplugin_b200.scenes import EMPTY_BVH
    p = scenes("entities")
    seeds = pass_seeds(4)
    load_scene(cuda_ctx, p)
    with_entities = _render(cuda_ctx, seeds)
    cuda_ctx.render_set_params(flags=native.CCU_RENDER_NO_ENTITIES)
    try:
        cuda_ctx.render_begin(p.width, p.height)
        got = _render(cuda_ctx, seeds)
        fh = cuda_ctx.first_hit(seeds[0])
    finally:
        cuda_ctx.render_set_params()
    bare = dataclasses.replace(p, world_bvh=EMPTY_BVH.copy(), actor_bvh=EMPTY_BVH.copy())
    o = oracle.Oracle(bare)
    assert np.array_equal(_bits(got), _bits(o.render(seeds)))
    assert not np.array_equal(_bits(got), _bits(with_entities))
    assert np.array_equal(fh["kind"], o.first_hit(seeds[0])["kind"]) and fh["kind"].max() == 1


def test_sunlight_off_is_the_scene_with_the_sun_flag_cleared(scenes, cuda_ctx):
    """CCU_RENDER_NO_SUN == sunData flags bit 0 = 0 (PackedSun.java:16; sky.h:45,69): no sun sampling, no sun disc."""
    import oracle
    from chunkyclplugin_b200 import native
    p = scenes("terrain256")
    assert int(p.sun[0]) & 1
    seeds = pass_seeds(3)
    load_scene(cuda_ctx, p)
    cuda_ctx.render_set_params(flags=native.CCU_RENDER_NO_SUN)
    try:
        got = _render(cuda_ctx, seeds)
    finally:
        cuda_ctx.render_set_params()
    sun = p.sun.copy()
    sun[0] &= ~1
    assert np.array_equal(_bits(got), _bits(oracle.Oracle(dataclasses.replace(p, sun=sun)).render(seeds)))
    with pytest.raises(native.ChunkyCuError):
        cuda_ctx.render_set_params(flags=64)            # unknown bits are refused
    with pytest.raises(native.ChunkyCuError):
        cuda_ctx.render_set_params(kernel=2)            # kernels 2 / 3 of round 1 are gone


def test_second_scene_does_not_inherit_the_first_scenes_entities(scenes, cuda_ctx):
    """ccu_scene_begin starts from nothing, like the reference's loader (fresh palettes and EMPTY_NODE BVHs per load,
    AbstractSceneLoader.java:70-140): a scene that sets no BVHs / models after a scene that did renders without them."""
    import oracle
    ent, ter = scenes("entities"), scenes("terrain128")
    seeds = pass_seeds(3)
    load_scene(cuda_ctx, ent)
    _render(cuda_ctx, seeds)
    ctx = cuda_ctx
    ctx.scene_begin()
    ctx.set_atlas(ter.atlas)
    ctx.set_block_palette(ter.block_palette)
    ctx.set_material_palette(ter.mat_palette)
    ctx.set_sun(ter.sun)
    ctx.set_sky(ter.sky, ter.sky_intensity)
    ctx.set_octree(ter.octree, ter.octree_depth)          # no models, no triangles, no BVHs
    ctx.scene_commit()
    ctx.camera_set(ter.projector_type, ter.camera)
    ctx.render_begin(ter.width, ter.height)
    got = _render(ctx, seeds)
    assert np.array_equal(_bits(got), _bits(oracle.Oracle(ter).render(seeds)))
    from chunkyclplugin_b200 import native
    ctx.scene_begin()
    with pytest.raises(native.ChunkyCuError):
        ctx.scene_commit()                                # the mandatory arrays of the previous scene are not inherited either


# ---------------------------------------------------------------------------------------------------------
# deep worlds / deep BVHs
# ---------------------------------------------------------------------------------------------------------
def test_deep_world_uses_nodes_between_top_table_and_bricks(scenes, cuda_ctx):
    """Octree depth 13: the top table cannot have 16^3 cells any more (air_cell_level 6, 64-ary nodes down to the bricks)."""
    import oracle
    from chunkyclplugin_b200 import native
    p = scenes("terrain128")
    deep = dataclasses.replace(p, octree=embed_octree(p.octree, 6), octree_depth=p.octree_depth + 6)
    assert deep.octree_depth == 13
    xyz = np.random.default_rng(1).integers(0, 128, size=(5000, 3))
    a = native.layout_lookup(p.octree, p.octree_depth, xyz)
    b = native.layout_lookup(deep.octree, deep.octree_depth, xyz)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    seeds = pass_seeds(3)
    load_scene(cuda_ctx, deep)
    got = _render(cuda_ctx, seeds)
    assert np.array_equal(_bits(got), _bits(oracle.Oracle(deep).render(seeds)))
    fh, rf = cuda_ctx.first_hit(seeds[0]), oracle.Oracle(deep).first_hit(seeds[0])
    assert np.array_equal(fh["node"], rf["node"]) and np.array_equal(_bits(fh["t"]), _bits(rf["t"]))
    cuda_ctx.render_set_params(kernel=1)
    try:
        cuda_ctx.render_begin(deep.width, deep.height)
        assert np.array_equal(_bits(_render(cuda_ctx, seeds)), _bits(got))
    finally:
        cuda_ctx.render_set_params()


def _chain_bvh(p, depth):
    """A degenerate world BVH: `depth` inner nodes in a chain, every right child the same small leaf, the last left child
    the scene's own BVH root re-based.  Valid for the reference (its stack only overflows with > 64 entries PENDING)."""
    from chunkyclplugin_b200.scenes import EMPTY_BVH
    bvh = np.asarray(p.world_bvh, np.int32)
    n_nodes = bvh.size // 7
    root_box = bvh[1:7].copy()
    # right child of every chain node: a leaf whose box (NaN bounds) no ray can enter, so nothing is ever left pending
    leaf = next(i for i in range(n_nodes) if bvh[7 * i] <= 0)
    leaf_node = np.concatenate([bvh[7 * leaf:7 * leaf + 1], EMPTY_BVH[1:7]]).astype(np.int32)
    # layout: chain node c at 14*c (7 ints) followed by ... the reference wants first child at node + 7, second child at node[0]
    # chain node c: [ptr to right child, box]; left child = next chain node at +7; right children stored after the chain + tree
    out = []
    base_tree = 7 * depth                 # original tree starts here (it is the left child of the last chain node)
    right_base = base_tree + bvh.size     # `depth` copies of the leaf node
    for c in range(depth):
        out.append(np.concatenate([[right_base + 7 * c], root_box]).astype(np.int32))
    tree = bvh.copy()
    for i in range(n_nodes):
        if tree[7 * i] > 0:
            tree[7 * i] += base_tree
    out.append(tree)
    for c in range(depth):
        out.append(leaf_node)
    return np.concatenate(out).astype(np.int32)


def test_bvh_deeper_than_the_reference_stack_still_renders(scenes, cuda_ctx):
    """A valid BVH 70 levels deep: the wavefront kernel's layout refuses it (explicit kernel 4 -> clear error), the default
    kernel selection falls back to the thread-per-pixel kernel on the reference's own arrays and renders it."""
    import oracle
    from chunkyclplugin_b200 import native
    p = scenes("entities")
    deep = dataclasses.replace(p, world_bvh=_chain_bvh(p, 70))
    seeds = pass_seeds(2)
    ref = oracle.Oracle(deep).render(seeds)
    load_scene(cuda_ctx, deep)
    got = _render(cuda_ctx, seeds)                      # kernel 0
    assert np.array_equal(_bits(got), _bits(ref))
    cuda_ctx.render_set_params(kernel=4)
    try:
        with pytest.raises(native.ChunkyCuError, match="BVH"):
            cuda_ctx.render_passes(np.asarray(seeds, np.int32))
    finally:
        cuda_ctx.render_set_params()


# ---------------------------------------------------------------------------------------------------------
# overlap: merge of window k with the passes of window k+1; camera-ray upload with the passes in flight
# ---------------------------------------------------------------------------------------------------------
def test_async_merge_racing_the_next_window_is_bit_identical(scenes, cuda_ctx):
    """ccu_render_merge_async returns while the read-back / merge runs; the next window renders into the second buffer.
    Same sample buffer as the blocking sequence (OpenClPathTracingRenderer.java:150-151,164-177)."""
    p = scenes("terrain256")
    seeds = pass_seeds(18)
    n = p.width * p.height * 3
    # blocking reference sequence
    load_scene(cuda_ctx, p)
    want = np.zeros(n, np.float64)
    spp = 0
    for lo, hi in ((0, 5), (5, 11), (11, 18)):
        cuda_ctx.render_passes(seeds[lo:hi])
        spp += cuda_ctx.render_merge(want, spp)
    assert spp == 18
    # overlapped sequence
    load_scene(cuda_ctx, p)
    got = np.zeros(n, np.float64)
    spp = 0
    for lo, hi in ((0, 5), (5, 11), (11, 18)):
        cuda_ctx.render_passes(seeds[lo:hi], block=False)          # queued behind nothing: the previous merge reads the other buffer
        spp += cuda_ctx.render_merge_async(got, spp)               # waits for the previous merge, closes this window, returns
    cuda_ctx.render_merge_wait()
    assert spp == 18
    assert np.array_equal(got, want)
    assert got.max() > 0


def test_window_close_then_merge_on_another_thread(scenes, cuda_ctx):
    """The two-call form the Java shim uses: close on the render thread, merge on a pool thread while the next window renders."""
    from chunkyclplugin_b200 import native
    p = scenes("terrain256")
    seeds = pass_seeds(12)
    n = p.width * p.height * 3
    load_scene(cuda_ctx, p)
    want = np.zeros(n, np.float64)
    cuda_ctx.render_passes(seeds[:6]); cuda_ctx.render_merge(want, 0)
    cuda_ctx.render_passes(seeds[6:]); cuda_ctx.render_merge(want, 6)
    load_scene(cuda_ctx, p)
    got = np.zeros(n, np.float64)
    cuda_ctx.render_passes(seeds[:6])
    assert cuda_ctx.render_window_close() == 6
    with pytest.raises(native.ChunkyCuError):
        cuda_ctx.render_read()                                     # the closed window owns the staging buffer
    t = threading.Thread(target=cuda_ctx.render_window_merge, args=(got, 0))
    t.start()
    cuda_ctx.render_passes(seeds[6:])                              # renders into the second buffer meanwhile
    t.join()
    assert cuda_ctx.render_window_close() == 6
    cuda_ctx.render_window_merge(got, 6)
    assert cuda_ctx.render_window_close() == 0                     # nothing open: nothing to merge
    assert np.array_equal(got, want)


def test_window_start_reads_the_previous_windows_mean(scenes, cuda_ctx):
    """With two window buffers the first pass of a window still sees what the reference's single buffer would hold
    (mean * 0 + colour, rayTracer.cl:111): an inf left by the previous window turns into NaN there, and here."""
    import oracle
    p = scenes("terrain64")
    seeds = pass_seeds(4)
    load_scene(cuda_ctx, p)
    cuda_ctx.render_passes(seeds[:2])
    sb = np.zeros(p.width * p.height * 3, np.float64)
    cuda_ctx.render_merge_async(sb, 0)
    cuda_ctx.render_passes(seeds[2:])
    cuda_ctx.render_merge_wait()
    got, spp = cuda_ctx.render_read()
    assert spp == 2
    o = oracle.Oracle(p)
    ref = o.render(seeds[:2])
    ref = o.render(seeds[2:], start_spp=0, res=ref)
    assert np.array_equal(_bits(got), _bits(ref))


def test_camera_rays_replaced_while_passes_are_in_flight(scenes, cuda_ctx):
    """projectorType -1: a new ray set uploaded during a batch (ClCamera.generate from the camera task,
    OpenClPathTracingRenderer.java:146-148) is used by the NEXT batch; the batch in flight keeps its rays."""
    import oracle
    from chunkyclplugin_b200.scenes import pregenerated_rays
    p = scenes("terrain256")
    rng = np.random.default_rng(3)
    rays = [pregenerated_rays(p.camera, p.width, p.height, jitter=rng) for _ in range(3)]
    q = [dataclasses.replace(p, projector_type=-1, camera=r) for r in rays]
    seeds = pass_seeds(9)
    load_scene(cuda_ctx, q[0])
    cuda_ctx.render_passes(seeds[0:3], block=False)
    cuda_ctx.camera_set(-1, rays[1])                     # uploads into the buffer no launch reads, on the copy stream
    cuda_ctx.render_passes(seeds[3:6], block=False)
    cuda_ctx.camera_set(-1, rays[2])
    cuda_ctx.render_passes(seeds[6:9], block=False)
    got, spp = cuda_ctx.render_read()
    assert spp == 9
    ref = None
    for i in range(3):
        ref = oracle.Oracle(q[i]).render(seeds[3 * i:3 * i + 3], start_spp=3 * i, res=ref)
    assert np.array_equal(_bits(got), _bits(ref))


def test_host_renderer_regenerates_jittered_rays(scenes):
    """CudaPathTracingRenderer with a generated-ray camera: rays are re-drawn between batches (ADVICE r1: frozen rays gave
    no anti-aliasing for non-pinhole projections), batches are capped, and the result is the mean over the ray sets used."""
    from chunkyclplugin_b200.renderer import CudaPathTracingRenderer, CudaSceneLoader, DefaultRenderManager, RendererInstance, Scene
    from chunkyclplugin_b200.scenes import pregenerated_rays
    p = scenes("terrain64")
    q = dataclasses.replace(p, projector_type=-1, camera=pregenerated_rays(p.camera, p.width, p.height))
    rng = np.random.default_rng(11)
    calls = []

    def gen(jitter):
        calls.append(jitter)
        return pregenerated_rays(p.camera, p.width, p.height, jitter=rng if jitter else None)

    inst = RendererInstance.get(0)
    scene = Scene(q, target_spp=24, ray_generator=gen)
    r = CudaPathTracingRenderer(CudaSceneLoader(inst), camera_regen_passes=4)
    r.render(DefaultRenderManager(scene))
    assert scene.spp == 24
    assert len(calls) >= 3 and all(calls)               # the initial set + regenerated sets, all jittered
    frozen = Scene(q, target_spp=24)
    CudaPathTracingRenderer(CudaSceneLoader(inst)).render(DefaultRenderManager(frozen))
    a, b = scene.sample_buffer.reshape(-1, 3), frozen.sample_buffer.reshape(-1, 3)
    assert np.isfinite(a).all() and a.max() > 0
    assert not np.array_equal(a, b)                     # different sub-pixel positions were sampled
    assert abs(a.mean() / b.mean() - 1.0) < 0.05        # ... of the same image
    RendererInstance.reset()


def test_render_sync_does_not_hold_the_context_lock(scenes, cuda_ctx):
    """While one thread waits for a long batch, another thread's calls on the same context go through (ADVICE r1:
    ccu_render_sync held the mutex for the whole batch)."""
    import time
    p = scenes("terrain256")
    load_scene(cuda_ctx, p)
    seeds = pass_seeds(3000)
    t_done = {}

    def waiter():
        cuda_ctx.render_passes(seeds)                   # blocking: async + sync
        t_done["render"] = time.perf_counter()

    t = threading.Thread(target=waiter)
    t0 = time.perf_counter()
    t.start()
    time.sleep(0.005)
    n = cuda_ctx.launch_count()                         # takes the context lock
    cuda_ctx.render_set_params()
    t_done["other"] = time.perf_counter()
    t.join()
    assert n > 0
    assert t_done["other"] < t_done["render"], (t_done["other"] - t0, t_done["render"] - t0)
