"""Inputs the parity scenes never produce, against the CPU oracle, bit-exact on every pixel of every output:

A. sky tables on both sides of the shared-memory staging threshold of the wavefront kernel,
B. BVH walks whose traversal stack grows past the 12 entries kept in shared memory,
C. canvases that are not multiples of the 32x32 pixel tiles of the thread-per-ray kernels,
D. texture atlases built the way the Java loader builds them (4096-wide layers, one write per texture).

The scene helpers live here; the tests without a `gpu` mark check the fixtures themselves on the CPU."""
import dataclasses

import numpy as np
import pytest

from chunkyclplugin_b200.javarandom import pass_seeds
from conftest import load_scene


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _render(ctx, p, seeds, kernel):
    """`seeds` passes with an explicit kernel (1 thread-per-pixel, 4 wavefront) into a fresh accumulation window."""
    ctx.render_set_params(kernel=kernel)
    try:
        ctx.render_begin(p.width, p.height)
        ctx.render_passes(np.asarray(seeds, np.int32))
        return ctx.render_read()[0]
    finally:
        ctx.render_set_params()


def _assert_first_hit_equal(got, want):
    for k in ("block", "face", "node", "kind"):
        assert np.array_equal(got[k], want[k]), k
    for k in ("t", "normal", "color"):
        assert np.array_equal(_bits(got[k]), _bits(want[k])), k


def _without_sun(p):
    sun = p.sun.copy()
    sun[0] &= ~1
    return dataclasses.replace(p, sun=sun)


# ---------------------------------------------------------------------------------------------------------
# A. sky tables
# ---------------------------------------------------------------------------------------------------------
def noise_sky(res, seed):
    """res x res RGBA8 sky table of hashed bytes: a lookup that reads any other texel sees another value."""
    from chunkyclplugin_b200.scenes import hash_u32
    j, i, c = np.meshgrid(np.arange(res), np.arange(res), np.arange(4), indexing="ij")
    return np.ascontiguousarray((hash_u32(j, i, c, seed) & 0xFF).astype(np.uint8))


def _sky_scene(scenes, variant, res):
    name, _, sun = variant.partition("_")
    p = dataclasses.replace(scenes(name), sky=noise_sky(res, seed=res))
    return _without_sun(p) if sun == "nosun" else p


@pytest.mark.gpu
@pytest.mark.parametrize("res", [1, 2, 3, 17, 63, 64, 65, 100, 128, 256])
@pytest.mark.parametrize("variant", ["terrain64", "mixed", "terrain64_nosun", "mixed_nosun"])
def test_sky_table_sizes(scenes, cuda_ctx, variant, res):
    """Sky resolution is a user setting (ClSky.java).  With the default 16 KiB threshold res <= 64 is staged in shared memory
    by the wavefront kernel - behind the top table on terrain64 (no BVH), behind the traversal stacks on mixed - and larger
    tables are read from global memory.  Without the sun every sky lookup is visible."""
    import oracle
    p = _sky_scene(scenes, variant, res)
    seeds = pass_seeds(3)
    o = oracle.Oracle(p)
    ref = o.render(seeds)
    load_scene(cuda_ctx, p)
    assert np.array_equal(_bits(_render(cuda_ctx, p, seeds, 4)), _bits(ref))
    assert np.array_equal(_bits(_render(cuda_ctx, p, seeds, 1)), _bits(ref))
    assert np.array_equal(cuda_ctx.preview(), o.preview())


# Largest staged tables with CCU_SKY_SMEM_MAX raised (ccu_queue.cuh: q_smem_bytes, Q_SMEM_LIMIT = 227 * 1024 - 1280 = 231168 B,
# 1024 slots, 4 bytes per texel).  Computed from the constants, not measured:
#   no BVH, top table staged:  (25 fields * 1024 + 4 stages * 32 mask words + 32 + 4096 top words) * 4 = 119424 B;
#                              (231168 - 119424) / 4 = 27936 texels -> 167^2 = 27889 fits, 168^2 = 28224 does not
#   BVH, top table staged:     (32 * 1024 + 7 * 32 + 32 + 4096 + 12 stack entries * 1024) * 4 = 197632 B;
#                              (231168 - 197632) / 4 = 8384 texels -> 91^2 = 8281 fits, 92^2 = 8464 does not
# large512 (depth 9) does not stage its top table (LAY 1): the sky starts right after the control words there.
@pytest.mark.gpu
@pytest.mark.parametrize("variant,res,knob", [
    ("terrain64", 64, "0"),               # below the default threshold, staging switched off: global path
    ("mixed", 64, "0"),
    ("terrain64", 167, "1048576"),        # the largest table that fits behind the top table
    ("terrain64", 168, "1048576"),        # one row more: global path
    ("mixed", 91, "1048576"),             # the largest table that fits behind the traversal stacks
    ("mixed", 92, "1048576"),
    ("large512", 64, None),               # top table not staged: the sky sits at a different offset
    ("large512", 100, "1048576"),
])
def test_sky_staging_threshold(scenes, cuda_ctx, monkeypatch, variant, res, knob):
    """CCU_SKY_SMEM_MAX moves the staging threshold (read at every launch); the image never changes."""
    import oracle
    p = _sky_scene(scenes, variant, res)
    seeds = pass_seeds(3)
    ref = oracle.Oracle(p).render(seeds)
    if knob is not None:
        monkeypatch.setenv("CCU_SKY_SMEM_MAX", knob)
    load_scene(cuda_ctx, p)
    assert np.array_equal(_bits(_render(cuda_ctx, p, seeds, 4)), _bits(ref))


# ---------------------------------------------------------------------------------------------------------
# B. deep traversal stacks
# ---------------------------------------------------------------------------------------------------------
def _leaf_texture(k):
    """16x16 RGBA8 leaf texture.  Every texture is transparent (alpha 0, which Material_sample rejects) in the same window of
    texels, so the terrain shows through all leaves there; textures with odd k also have hashed holes elsewhere."""
    from chunkyclplugin_b200.scenes import hash_u32
    y, x = np.mgrid[0:16, 0:16]
    h = hash_u32(x, y, k, 77)
    tex = np.zeros((16, 16, 4), np.uint8)
    for c in range(3):
        tex[..., c] = 40 + ((h >> (8 * c)) & 0x7F) + 40 * ((k + c) % 3)
    opaque = ~((x >= 3) & (x < 7) & (y >= 8) & (y < 13))
    if k % 2:
        opaque &= ((h >> 24) & 3) != 0
    tex[..., 3] = np.where(opaque, 255, 0)
    return tex


def _ray_slopes(p):
    """Extents of d.x / d.z and d.y / d.z over the primary rays of the canvas (pixel corners included), from the camera."""
    cam = np.asarray(p.camera, np.float64)
    m = cam[3:12].reshape(3, 3)
    x = (np.array([0.0, p.width]) - p.width / 2.0) / p.height
    y = np.array([-0.5, 0.5])
    xx, yy = np.meshgrid(x, y)
    d = np.stack([cam[14] * xx, cam[14] * yy, np.ones_like(xx)], axis=-1).reshape(-1, 3) @ m.T
    assert (d[:, 2] > 0.2).all()          # every primary ray travels towards +z
    sx, sy = d[:, 0] / d[:, 2], d[:, 1] / d[:, 2]
    return sx.min(), sx.max(), sy.min(), sy.max()


def nested_chain_bvh(p, depth):
    """`p` with a world BVH of `depth` inner nodes in a chain, walked down to the bottom by every primary ray with a pending
    entry left at every level.

    Chain node c: first child = chain node c + 1 (the last chain node: leaf A), second child = leaf c.  Every leaf holds one
    double-sided triangle in the plane z = camera z + dz that covers the whole view; its box is that triangle's box, so every
    primary ray enters it (at t > 0).  A chain node's box encloses the camera and everything below it, so the ray starts
    inside it (t < 0) and takes the chain first, pushing leaf c (bvh.h:93-108).  Deeper leaves lie nearer.  The deepest
    leaves are at node depth `depth`, what the layout's depth limit counts (ccu_layout.h bvh_ref).

    The triangles are similar in the camera's slope space, so a ray sees the same texel of each of them: the transparent
    window of _leaf_texture lets primary rays through all leaves to the terrain, and paths leave from leaves and terrain.
    Returns the new scene (triangles appended to the palette, textures to free atlas tiles, materials to the palette)."""
    from chunkyclplugin_b200.scenes import f2i, pack_material, pack_triangles
    sx0, sx1, sy0, sy1 = _ray_slopes(p)
    mx, my = 0.05 * (sx1 - sx0), 0.05 * (sy1 - sy0)
    lx, ly = 2 * (sx1 - sx0) + 4 * mx, 2 * (sy1 - sy0) + 4 * my
    corner = np.array([sx0 - mx, sy0 - my])
    cam = np.asarray(p.camera[0:3], np.float64)

    # textures on free tiles of the atlas, one material each
    atlas = p.atlas.copy()
    mats = p.mat_palette.tolist()
    leaf_mats = []
    for k in range(4):
        tx, ty = 12 + k, 12
        assert not atlas[0, ty * 16:ty * 16 + 16, tx * 16:tx * 16 + 16].any()
        atlas[0, ty * 16:ty * 16 + 16, tx * 16:tx * 16 + 16] = _leaf_texture(k)
        leaf_mats.append(len(mats))
        mats += pack_material((16 << 16) | 16, (tx << 22) | (ty << 13))

    def triangle(dz):
        s = [corner, corner + [lx, 0.0], corner + [0.0, ly]]
        return np.array([[cam[0] + a * dz, cam[1] + b * dz, cam[2] + dz] for a, b in s])

    # leaf c at dz(c), leaf A (index depth) nearest of all
    dz = 0.6 + 0.05 * (depth - np.arange(depth + 1))
    dz[depth] = 0.55
    tris = np.stack([triangle(z) for z in dz])
    material = np.array([leaf_mats[c % 4] for c in range(depth + 1)])
    packed = pack_triangles(tris, material, np.ones(depth + 1, bool))
    base = int(p.bvh_trigs.size)
    trigs = np.concatenate([p.bvh_trigs] + [np.concatenate([[1], packed[c]]) for c in range(depth + 1)]).astype(np.int32)
    leaf_ptr = base + 21 * np.arange(depth + 1)

    lo = tris.min(axis=1).astype(np.float32)
    hi = tris.max(axis=1).astype(np.float32)
    lo = np.where(lo.astype(np.float64) > tris.min(axis=1), np.nextafter(lo, np.float32(-np.inf)), lo)
    hi = np.where(hi.astype(np.float64) < tris.max(axis=1), np.nextafter(hi, np.float32(np.inf)), hi)

    def box(l, h):
        return list(f2i([l[0], h[0], l[1], h[1], l[2], h[2]]))

    # chain node c's box: the camera and leaves c .. depth, with a margin
    nodes = []
    for c in range(depth):
        l = np.minimum(lo[c:].min(axis=0), cam) - 1.0
        h = np.maximum(hi[c:].max(axis=0), cam) + 1.0
        nodes.append([7 * (depth + 1 + c)] + box(l, h))
    nodes.append([-int(leaf_ptr[depth])] + box(lo[depth], hi[depth]))            # leaf A at 7 * depth
    for c in range(depth):
        nodes.append([-int(leaf_ptr[c])] + box(lo[c], hi[c]))                    # leaf c at 7 * (depth + 1 + c)
    world = np.array(nodes, np.int64).astype(np.int32).reshape(-1)
    return dataclasses.replace(p, world_bvh=world, bvh_trigs=trigs, atlas=atlas, mat_palette=np.asarray(mats, np.int32))


def _first_descent_pending(p, seed):
    """bvh.h:22-113 restated for the camera rays of `seed`, up to the first leaf each walk reaches: the number of pending
    nodes (toVisit) there.  The walk starts with the distance the octree left (the scene without BVHs), as closestIntersect
    runs the octree first (kernel.h:14-24); before the first leaf no triangle can shorten it, so the count is exact."""
    import oracle
    from chunkyclplugin_b200.scenes import EMPTY_BVH
    bare = dataclasses.replace(p, world_bvh=EMPTY_BVH.copy(), actor_bvh=EMPTY_BVH.copy())
    dist = oracle.Oracle(bare).first_hit(seed)["t"]
    rays = oracle.Oracle(p).camera_rays(seed)
    bvh = np.asarray(p.world_bvh, np.int32)
    boxes = bvh.view(np.float32)
    pick = np.random.default_rng(seed & 0xFFFF).choice(rays.shape[0], size=min(300, rays.shape[0]), replace=False)
    out = []
    with np.errstate(divide="ignore", invalid="ignore"):
        for i in pick:
            o, d = rays[i, 0:3], rays[i, 3:6]
            inv = np.float32(1.0) / d

            def entry(node):
                b = boxes[node + 1:node + 7]
                t1 = (b[0::2] - o) * inv
                t2 = (b[1::2] - o) * inv
                tmin = np.fmax(np.fmax(np.fmin(t1[0], t2[0]), np.fmin(t1[1], t2[1])), np.fmin(t1[2], t2[2]))
                tmax = np.fmin(np.fmin(np.fmax(t1[0], t2[0]), np.fmax(t1[1], t2[1])), np.fmax(t1[2], t2[2]))
                return np.float32(np.nan) if tmax < tmin else tmin

            cur, pending = 0, 0
            while bvh[cur] > 0:
                off = int(bvh[cur])
                t1, t2 = entry(cur + 7), entry(off)
                miss1 = np.isnan(t1) or t1 > dist[i]
                miss2 = np.isnan(t2) or t2 > dist[i]
                if miss1 and miss2:
                    break                       # nothing pending is deeper than here
                if miss1:
                    cur = off
                elif miss2:
                    cur += 7
                else:
                    pending += 1
                    cur = cur + 7 if t1 < t2 else off
            out.append(pending)
    return np.array(out)


@pytest.mark.parametrize("depth", [13, 40, 63])
def test_nested_chain_bvh_fills_the_traversal_stack(scenes, depth):
    """The fixture does what part B relies on: primary rays reach a leaf with about `depth` nodes pending, past the 12
    stack entries the wavefront kernel keeps in shared memory."""
    p = nested_chain_bvh(scenes("entities"), depth)
    pending = _first_descent_pending(p, pass_seeds(1)[0])
    assert pending.max() > 12
    if depth >= 40:
        assert pending.max() >= depth - 1
        assert (pending >= depth - 1).mean() > 0.5


def test_bvh_layout_depth_limit():
    """The commit-time layout holds a BVH whose deepest leaf is at node depth 63 and refuses depth 64 (the 64 entries of the
    reference's traversal stack, bvh.h:38)."""
    from chunkyclplugin_b200 import native
    from chunkyclplugin_b200 import scenes as S
    p = S.terrain_scene(8, 16, 9, seed=3)
    for depth, ok in ((63, True), (64, False)):
        q = nested_chain_bvh(p, depth)
        assert native.debug_bvh_layout(q.world_bvh, q.bvh_trigs)[3] is ok, depth


@pytest.mark.gpu
@pytest.mark.parametrize("depth", [11, 12, 13, 40, 63])
def test_deep_bvh_walks(scenes, cuda_ctx, depth):
    """Walks that leave `depth` nodes pending, shadow rays that end on the first accepted triangle with entries still on the
    stack, and the actor BVH walked after them: kernel 4, kernel 1 and the first hit against the oracle."""
    import oracle
    p = nested_chain_bvh(scenes("entities"), depth)
    seeds = pass_seeds(2)
    o = oracle.Oracle(p)
    ref = o.render(seeds)
    load_scene(cuda_ctx, p)
    assert np.array_equal(_bits(_render(cuda_ctx, p, seeds, 4)), _bits(ref))
    assert np.array_equal(_bits(_render(cuda_ctx, p, seeds, 1)), _bits(ref))
    fh, want = cuda_ctx.first_hit(seeds[0]), o.first_hit(seeds[0])
    _assert_first_hit_equal(fh, want)
    assert (want["kind"] == 2).mean() > 0.3 and (want["kind"] == 1).any()      # leaves in front, terrain through the window


@pytest.mark.gpu
def test_deep_bvh_walks_in_every_slot(scenes, cuda_ctx):
    """At least one pixel per slot of every CTA (sm_count x 1024): every CTA's part of the global stack scratch is used."""
    import oracle
    from chunkyclplugin_b200 import native
    sms = native.device_info(0)["sm_count"]
    w = 480
    h = -(-sms * 1024 // w)
    p = nested_chain_bvh(dataclasses.replace(scenes("entities"), width=w, height=h), 40)
    assert p.width * p.height >= sms * 1024
    seeds = pass_seeds(1)
    ref = oracle.Oracle(p).render(seeds)
    load_scene(cuda_ctx, p)
    assert np.array_equal(_bits(_render(cuda_ctx, p, seeds, 4)), _bits(ref))


@pytest.mark.gpu
def test_bvh_depth_64_falls_back_to_the_reference_arrays(scenes, cuda_ctx):
    """Depth 64 is more than the wavefront kernel's layout holds: kernel 4 refuses it, the default kernel renders it."""
    import oracle
    from chunkyclplugin_b200 import native
    p = nested_chain_bvh(scenes("entities"), 64)
    seeds = pass_seeds(2)
    load_scene(cuda_ctx, p)
    with pytest.raises(native.ChunkyCuError, match="BVH"):
        _render(cuda_ctx, p, seeds, 4)
    assert np.array_equal(_bits(_render(cuda_ctx, p, seeds, 0)), _bits(oracle.Oracle(p).render(seeds)))


# ---------------------------------------------------------------------------------------------------------
# C. canvas shapes for the thread-per-ray kernels
# ---------------------------------------------------------------------------------------------------------
CANVASES = [(1, 1), (8, 4), (31, 33), (33, 31), (37, 70), (97, 45), (257, 3), (3, 257)]


def _check_canvas(ctx, p, seeds):
    import oracle
    o = oracle.Oracle(p)
    load_scene(ctx, p)
    _assert_first_hit_equal(ctx.first_hit(seeds[0]), o.first_hit(seeds[0]))
    assert np.array_equal(ctx.preview(), o.preview())
    ref = o.render(seeds)
    assert np.array_equal(_bits(_render(ctx, p, seeds, 1)), _bits(ref))
    assert np.array_equal(_bits(_render(ctx, p, seeds, 4)), _bits(ref))


@pytest.fixture(scope="module")
def ctx_no_wide():
    """A context of its own for scenes committed with CCU_NO_WIDE (the reference's arrays, layout mode 0)."""
    from chunkyclplugin_b200 import native
    ctx = native.Context(0)
    yield ctx
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("wh", CANVASES)
@pytest.mark.parametrize("name", ["terrain64", "mixed"])
def test_canvas_shapes(scenes, cuda_ctx, ctx_no_wide, monkeypatch, name, wh):
    """k_first_hit and k_preview hand pixels out in 32x32 tiles with 8x4 patches inside full tiles (tile_order_xy<true>);
    the right-hand and bottom tiles are narrower here.  Also kernel 1 and kernel 4, and the first hit without the commit-time
    layouts (k_first_hit<0, ...>).  mixed has both BVHs and a depth-of-field camera."""
    import oracle
    p = dataclasses.replace(scenes(name), width=wh[0], height=wh[1])
    seeds = pass_seeds(3)
    _check_canvas(cuda_ctx, p, seeds)
    monkeypatch.setenv("CCU_NO_WIDE", "1")
    load_scene(ctx_no_wide, p)
    _assert_first_hit_equal(ctx_no_wide.first_hit(seeds[0]), oracle.Oracle(p).first_hit(seeds[0]))


@pytest.mark.gpu
def test_canvas_shape_with_generated_rays(scenes, cuda_ctx):
    """projectorType -1 (one uploaded ray per pixel) on a canvas with partial tiles on both edges."""
    from chunkyclplugin_b200.scenes import pregenerated_rays
    p = scenes("terrain64")
    w, h = 97, 45
    rays = pregenerated_rays(p.camera, w, h, jitter=np.random.default_rng(5))
    _check_canvas(cuda_ctx, dataclasses.replace(p, projector_type=-1, camera=rays, width=w, height=h), pass_seeds(3))


# ---------------------------------------------------------------------------------------------------------
# D. atlases as the Java loader builds them
# ---------------------------------------------------------------------------------------------------------
def _texture(w, h, salt, cut=False):
    """w x h RGBA8 texture of hashed colours; `cut`: a quarter of the texels transparent."""
    from chunkyclplugin_b200.scenes import hash_u32
    y, x = np.mgrid[0:h, 0:w]
    v = hash_u32(x, y, salt, 5)
    tex = np.stack([(v >> s) & 0xFF for s in (0, 8, 16)] + [np.full_like(v, 255)], axis=-1).astype(np.uint8)
    if cut:
        tex[..., 3] = np.where(((v >> 24) & 3) == 0, 0, 255)
    return tex


def java_atlas(width, height, layers, placed):
    """Textures placed as CudaTextureLoader does: `placed` = [(tile_x, tile_y, layer, rgba)] on the 16-texel tile grid.
    Returns the writes (x, y, layer, rgba) of one ccu_scene_atlas_write each, the dense (layers, height, width, 4) array the
    oracle reads, and per texture its record (size = w << 16 | h, location = x << 22 | y << 13 | layer, ClTextureLoader.java:123-132)."""
    writes, records = [], []
    dense = np.zeros((layers, height, width, 4), np.uint8)
    for tx, ty, layer, rgba in placed:
        h, w = rgba.shape[:2]
        x, y = 16 * tx, 16 * ty
        assert x + w <= width and y + h <= height and layer < layers
        writes.append((x, y, layer, rgba))
        dense[layer, y:y + h, x:x + w] = rgba
        records.append(((w << 16) | h, (tx << 22) | (ty << 13) | layer))
    return writes, dense, records


# decorated terrain64: 8 textured materials (stone, dirt, grass, sand, glowstone, glass, slab, cross - Palettes order) + sun
ATLASES = {
    # 4096 x 64 x 3: tile x 0, 15, 16 and 255; 8x8, 16x16, 32x32, 64x16, 16x64; tile y > 0 on layers 1 and 2 (their layer
    # field overlaps tile y and clamps to the last layer, SURVEY Q9).  The last entry is not a material: it sits where the
    # clamped glass record reads (layer 2 instead of 1).
    "java4096x64x3": (4096, 64, 3, [
        (0, 0, 0, (16, 16)), (15, 0, 0, (8, 8)), (16, 0, 0, (16, 16)), (255, 0, 0, (16, 16)), (100, 0, 1, (16, 64)),
        (40, 1, 1, (32, 32)), (200, 2, 2, (64, 16)), (3, 1, 2, (16, 16)), (17, 0, 0, (32, 32)), (40, 1, 2, (32, 32))]),
    # 4090 x 40 x 1: extents that are not tile multiples; grass is a 10x8 texture ending at the last column and row, and its
    # material claims 16x16 (4th field), so its reads clamp at both atlas edges
    "odd4090x40": (4090, 40, 1, [
        (0, 0, 0, (16, 16)), (254, 0, 0, (16, 16)), (255, 2, 0, (10, 8), (16, 16)), (100, 0, 0, (32, 32)), (7, 1, 0, (8, 8)),
        (5, 1, 0, (16, 16)), (200, 1, 0, (64, 16)), (9, 0, 0, (16, 16)), (10, 0, 0, (32, 32))]),
}


def _java_atlas_scene(p, name):
    """`p` (decorated terrain64) with its textures moved to the placements of ATLASES[name]."""
    width, height, layers, spec = ATLASES[name]
    placed = [(tx, ty, l, _texture(w, h, salt=i, cut=i in (5, 7))) for i, (tx, ty, l, (w, h), *_) in enumerate(spec)]
    writes, dense, records = java_atlas(width, height, layers, placed)
    for i, entry in enumerate(spec):
        if len(entry) == 5:                      # the material claims another size than the texture written
            w, h = entry[4]
            records[i] = ((w << 16) | h, records[i][1])
    mats = p.mat_palette.copy().reshape(-1, 6)
    textured = np.nonzero(mats[:, 0] & 4)[0]
    assert textured.size == 8
    for m, (size, loc) in zip(textured, records):
        mats[m, 2], mats[m, 3] = size, loc
    sun = p.sun.copy()
    sun[1], sun[2] = records[8]
    q = dataclasses.replace(p, atlas=dense, mat_palette=mats.reshape(-1), sun=sun)
    return q, writes, mats[textured, 3]


def _load_with_writes(ctx, p, writes, atlas):
    ctx.scene_begin()
    ctx.atlas_create(atlas.shape[2], atlas.shape[1], atlas.shape[0])
    for x, y, layer, rgba in writes:
        ctx.atlas_write(x, y, layer, rgba)
    ctx.set_block_palette(p.block_palette)
    ctx.set_material_palette(p.mat_palette)
    ctx.set_aabb_models(p.aabb_models)
    ctx.set_quad_models(p.quad_models)
    ctx.set_triangles(p.bvh_trigs)
    ctx.set_world_bvh(p.world_bvh)
    ctx.set_actor_bvh(p.actor_bvh)
    ctx.set_sun(p.sun)
    ctx.set_sky(p.sky, p.sky_intensity)
    ctx.set_octree(p.octree, p.octree_depth)
    ctx.scene_commit()
    ctx.camera_set(p.projector_type, p.camera)
    ctx.render_begin(p.width, p.height)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(ATLASES))
def test_atlas_written_texture_by_texture(scenes, cuda_ctx, name):
    """One ccu_scene_atlas_write per texture into the tile-linear atlas gives what the oracle reads from the dense array,
    and the same as ccu_scene_set_atlas of that array."""
    import oracle
    p, writes, locations = _java_atlas_scene(scenes("decorated"), name)
    layers = p.atlas.shape[0]
    if layers > 1:
        assert ((locations & 0x7FFFF) >= layers).any()          # at least one record's layer field clamps (SURVEY Q9)
    seeds = pass_seeds(3)
    o = oracle.Oracle(p)
    ref = o.render(seeds)
    _load_with_writes(cuda_ctx, p, writes, p.atlas)
    got = _render(cuda_ctx, p, seeds, 0)
    assert np.array_equal(_bits(got), _bits(ref))
    want = o.first_hit(seeds[0])
    _assert_first_hit_equal(cuda_ctx.first_hit(seeds[0]), want)
    assert np.array_equal(cuda_ctx.preview(), o.preview())
    assert len(np.unique(want["block"][want["kind"] == 1])) >= 4                # several of the moved textures are on screen
    load_scene(cuda_ctx, p)
    assert np.array_equal(_bits(_render(cuda_ctx, p, seeds, 0)), _bits(got))


@pytest.mark.gpu
def test_atlas_write_refuses_writes_outside_the_atlas(cuda_ctx):
    from chunkyclplugin_b200 import native
    tex = _texture(16, 16, salt=1)
    cuda_ctx.scene_begin()
    with pytest.raises(native.ChunkyCuError):
        cuda_ctx.atlas_write(0, 0, 0, tex)                      # before ccu_scene_atlas_create
    cuda_ctx.atlas_create(4090, 40, 2)
    cuda_ctx.atlas_write(4074, 24, 1, tex)                      # ends at the last column and row of the last layer
    for x, y, layer in ((4075, 0, 0), (0, 25, 0), (0, 0, 2), (-1, 0, 0), (0, -1, 0), (0, 0, -1)):
        with pytest.raises(native.ChunkyCuError):
            cuda_ctx.atlas_write(x, y, layer, tex)
