"""Every render kernel instance, run: the 120 k_render_queue<HAS_BVH, LAY, Shade> and 60 k_render_mega<MODE, Shade> of DESIGN §5,
each on a scene where every switch of its Shade changes the image, checked against the CPU restatement (FlagsOracle) bit for
bit and against the instance the launch reports (ccu_debug_last_render).  Also the selection rules of shade_variant on 16 small
scenes with each scene fact on or off, and the sky-staging boundary of every shared-memory footprint of the wavefront kernel.

The tests without a `gpu` mark check the fixtures themselves on the CPU: every switch acts, the cases cover every instance."""
import dataclasses
import functools
import itertools
import math

import numpy as np
import pytest

from chunkyclplugin_b200 import native
from chunkyclplugin_b200 import scenes as S
from chunkyclplugin_b200.javarandom import pass_seeds
from chunkyclplugin_b200.renderer import upload_scene
from oracle import edge_rays as E
from test_gpu_input_edges import noise_sky
from test_gpu_specular import assert_bits

import specular_oracle as SO

NO_ENTITIES, SPEC, NEE, NEAR, MODELS, BIOME = 1, 4, 8, 128, 256, 512
NEE_FLAGS = (0, NEE, NEE | NEAR, NEE | MODELS, NEE | NEAR | MODELS)   # indexed by NeeKind: none, area, near, area / near + models
# Shade i of the library's enumeration (nth_shade in chunkycu.cu): (spec, nee, biome)
SHADES = [(i % 2, i // 2 % 5, i // 10) for i in range(20)]
SEEDS = pass_seeds(3)
TORCH, LANTERN = 9, 10          # type indices the fixture appends to the mixed scene's palettes


def shade_flags(spec, nee, biome):
    """The render flags that select Shade<spec, nee, biome> on a scene that has everything."""
    return (SPEC if spec else 0) | NEE_FLAGS[nee] | (BIOME if biome else 0)


def shade_id(i):
    spec, nee, biome = SHADES[i]
    return ("spec" if spec else "plain") + "-" + ("none", "area", "near", "models", "nearmodels")[nee] + ("-biome" if biome else "")


# ---------------------------------------------------------------------------------------------------------
# shared-memory footprints of k_render_queue (ccu_queue.cuh: QField, q_smem_bytes, Q_SMEM_LIMIT)
# ---------------------------------------------------------------------------------------------------------
Q_SLOTS, Q_TOP_WORDS, Q_STACK_WORDS = 1024, 4096, 12 * 1024
Q_SMEM_LIMIT = 227 * 1024 - 1280          # 231168 B
SKY_SMEM_DEFAULT = 16384                  # CCU_SKY_SMEM_MAX unset


def q_smem_bytes(bvh, tops, spec, nee):
    """Dynamic shared memory of a launch before the sky table: 25 slot fields (32 with BVHs, 33 with BVHs and spec, 2 more with
    NEE) x 1024 slots, 4 (7 with BVHs) stage masks of 32 words, 32 control words, the staged top table, the BVH stacks."""
    fields = (33 if spec else 32) if bvh else 25
    fields += 2 if nee else 0
    return (fields * Q_SLOTS + (7 if bvh else 4) * 32 + 32 + (Q_TOP_WORDS if tops else 0) + (Q_STACK_WORDS if bvh else 0)) * 4


def staged_texels(bvh, tops, spec, nee, sky_res, sky_max=SKY_SMEM_DEFAULT):
    """The sky texels a kernel-4 launch stages in shared memory (chunkycu.cu, render_passes_locked)."""
    n = sky_res * sky_res
    return n if n * 4 <= sky_max and q_smem_bytes(bvh, tops, spec, nee) + n * 4 <= Q_SMEM_LIMIT else 0


# the 12 footprints: spec adds a slot field only with BVHs
FOOTPRINTS = [(bvh, tops, spec, nee) for bvh in (0, 1) for tops in (1, 0) for spec in ((0, 1) if bvh else (0,)) for nee in (0, 1)]


def largest_staged_sky(fp):
    return math.isqrt((Q_SMEM_LIMIT - q_smem_bytes(*fp)) // 4)


# ---------------------------------------------------------------------------------------------------------
# the variant fixture
# ---------------------------------------------------------------------------------------------------------
def _contact_stage(vox):
    """A sand floor in front of the camera with a sand block right below it that carries one glowstone and one lantern next to
    each other: the camera sees the surfaces within 1/8 of both from close by.  The terrain's glowstone within 40 voxels of the
    camera's z goes, so that the emitter lists around the stage hold few entries and the near-field samplers run often."""
    glow = vox == S.GLOWSTONE
    glow[:, :, 40:] = False
    vox[glow] = S.AIR
    vox[24:41, :21, 6:16] = S.SAND
    vox[24:41, 21:, 6:16] = S.AIR
    vox[28:37, :28, 5:8] = S.SAND
    vox[28:37, 28:, 5:8] = S.AIR
    vox[33, 28, 6] = S.GLOWSTONE
    vox[31, 28, 6] = LANTERN
    # model emitters of both kinds farther off, where the camera sees the terrain
    for x, z, block in ((20, 50, TORCH), (44, 56, TORCH), (30, 46, LANTERN)):
        vox[x, int(np.nonzero(vox[x, :, z])[0].max()) + 1, z] = block


@functools.lru_cache(maxsize=None)
def variant_scene(bvh: bool) -> S.PackedScene:
    """mixed_test_scene (models, alpha tests, both BVHs, DoF camera) with everything a Shade switch acts on: glossy materials
    (specular words), glowstone (full-cube emitters), torches and lanterns (model emitters, flat-coloured), biome colours over
    every chunk with grass- and water-tinted materials, and the contact stage.  bvh = False: both BVHs are EMPTY_BVH."""
    size = 64
    p = S.mixed_test_scene(size)
    full = S.terrain_voxels(0, 0, size, 256, size, seed=99, decorate=True)     # terrain_scene's voxels for size < 128
    shift = 64 - size // 3
    vox = np.ascontiguousarray(full[:, shift:shift + size, :])
    bp, mp = list(p.block_palette), list(p.mat_palette)
    quads, aabbs = list(p.quad_models), list(p.aabb_models)
    assert len(bp) == 2 * TORCH
    mat = len(mp)
    mp += S.pack_material(0, 0, textured=False, argb=S._s32(0xFFFFD070), emittance=1.0)
    mp += S.pack_material(0, 0, textured=False, argb=S._s32(0xFF404048))
    bp += [3, len(quads), 2, len(aabbs)]
    quads += S._torch_quads(mat)
    aabbs += S._lantern_boxes(mat, mat + 6)
    _contact_stage(vox)
    tree, depth = S.build_octree(vox, np.arange(LANTERN + 1, dtype=np.int64) * 2)
    q = dataclasses.replace(p, octree=tree, octree_depth=depth, block_palette=S._i32(bp), mat_palette=S._i32(mp),
                            quad_models=S._i32(quads), aabb_models=S._i32(aabbs), name="variants")
    q = S.with_biomes(S.water_tinted(S.glossy(q)), seed=5, holes=0.0)
    if not bvh:
        q = dataclasses.replace(q, world_bvh=S.EMPTY_BVH.copy(), actor_bvh=S.EMPTY_BVH.copy(), name=q.name + "_nobvh")
    return q


def deep(p):
    """p in the low corner of a depth-13 world (layout 2); entities and biome chunks keep their coordinates."""
    return dataclasses.replace(p, octree=E.embed_octree(p.octree, 13 - p.octree_depth), octree_depth=13, name=p.name + "_deep13")


_images = {}


def oracle_image(bvh: bool, flags: int) -> np.ndarray:
    """FlagsOracle's image of the variant scene: one per BVH state and flag set serves every layout."""
    key = (bool(bvh), flags)
    if key not in _images:
        _images[key] = SO.FlagsOracle(variant_scene(bvh), flags).render(SEEDS)
    return _images[key]


# single-switch steps between NEE flag sets: none <-> area, area <-> near, area <-> models, models <-> near models,
# near <-> near models
NEE_STEPS = [(0, 1), (1, 2), (1, 3), (3, 4), (2, 4)]
MIN_CHANGED = 0.01       # a switch changes at least this share of the pixels (measured minimum on the fixture: 1.5 %)


def _changed(a, b):
    return float(np.mean(~E.same_bits_or_nan(a, b).reshape(-1, 3).all(1)))


@pytest.mark.parametrize("bvh", [1, 0], ids=["bvh", "nobvh"])
def test_every_switch_acts_on_the_fixture(bvh):
    imgs = {i: oracle_image(bvh, shade_flags(*SHADES[i])) for i in range(20)}
    for i, j in itertools.combinations(range(20), 2):
        assert not E.same_bits_or_nan(imgs[i], imgs[j]).all(), (shade_id(i), shade_id(j))
    steps = []
    for spec, nee, biome in itertools.product((0, 1), range(5), (0, 1)):
        steps += [((spec, nee, biome), (1, nee, biome))] if not spec else []
        steps += [((spec, nee, biome), (spec, nee, 1))] if not biome else []
        steps += [((spec, a, biome), (spec, b, biome)) for a, b in NEE_STEPS if a == nee]
    assert len(steps) == 10 + 10 + 4 * 5
    for a, b in steps:
        got = _changed(oracle_image(bvh, shade_flags(*a)), oracle_image(bvh, shade_flags(*b)))
        assert got >= MIN_CHANGED, (a, b, got)


def test_fixture_has_what_every_switch_needs():
    for bvh in (0, 1):
        p = variant_scene(bvh)
        assert (p.mat_palette[5::6] != 0).any()
        assert SO.emitter_grid(p)["has_emitters"] and SO.emitter_grid(p, models=True)["has_emitters"]
        assert p.biome is not None and p.biome[0].shape[0] == 16
        assert (p.world_bvh.size > 7) == bool(bvh)


def test_deep_world_renders_as_the_shallow_one():
    """One oracle image per BVH state serves the depth-13 layout: the embedded scene renders the same bits."""
    flags = SPEC | NEE | NEAR | MODELS | BIOME
    for bvh in (0, 1):
        p = deep(variant_scene(bvh))
        assert_bits(SO.FlagsOracle(p, flags).render(SEEDS), oracle_image(bvh, flags))


# ---------------------------------------------------------------------------------------------------------
# the instance matrix
# ---------------------------------------------------------------------------------------------------------
# (kernel, has_bvh, lay or mode, shade): kernel 4 x HAS_BVH x LAY x 20, kernel 1 x MODE x 20 (on the BVH scene)
CASES = ([(4, bvh, lay, i) for bvh in (1, 0) for lay in (0, 1, 2) for i in range(20)]
         + [(1, 1, mode, i) for mode in (0, 1, 2) for i in range(20)])


def _case_id(c):
    kernel, bvh, lay, i = c
    return (f"k4-{'bvh' if bvh else 'nobvh'}-lay{lay}" if kernel == 4 else f"k1-mode{lay}") + "-" + shade_id(i)


def test_the_cases_cover_every_instance():
    queue = {(4, bvh, lay, SHADES[i]) for kernel, bvh, lay, i in CASES if kernel == 4}
    mega = {(1, mode, SHADES[i]) for kernel, _, mode, i in CASES if kernel == 1}
    assert len(CASES) == 180 and len(queue) == 120 and len(mega) == 60
    assert len(set(SHADES)) == 20


def test_footprint_arithmetic():
    """The footprints restated here agree with the numbers ccu_queue.cuh, DESIGN §10 and test_gpu_input_edges state."""
    assert q_smem_bytes(0, 1, 0, 0) == 119424 and largest_staged_sky((0, 1, 0, 0)) == 167
    assert q_smem_bytes(1, 1, 0, 0) == 197632 and largest_staged_sky((1, 1, 0, 0)) == 91
    assert q_smem_bytes(1, 1, 1, 1) == 209920 and largest_staged_sky((1, 1, 1, 1)) == 72
    assert q_smem_bytes(1, 1, 1, 1) + 64 * 64 * 4 == 226304
    assert len(set(FOOTPRINTS)) == 12
    for fp in FOOTPRINTS:
        r = largest_staged_sky(fp)
        assert staged_texels(*fp, r, 1 << 20) == r * r and staged_texels(*fp, r + 1, 1 << 20) == 0
        assert staged_texels(*fp, 64) == 64 * 64 and staged_texels(*fp, 65) == 0


@pytest.fixture(scope="module")
def ctx_no_wide():
    """A context of its own for scenes committed with CCU_NO_WIDE (the reference's arrays, layout mode 0)."""
    ctx = native.Context(0)
    yield ctx
    ctx.close()


@pytest.fixture(scope="module")
def loader():
    """Uploads a scene (with its biome colours) unless the context already holds it from this module."""
    held = {}

    def load(ctx, p, key):
        if held.get(id(ctx)) != key:
            held[id(ctx)] = None
            upload_scene(ctx, p)
            held[id(ctx)] = key
        ctx.camera_set(p.projector_type, p.camera)
        return ctx

    return load


def _render(ctx, p, seeds, kernel, flags):
    ctx.render_set_params(kernel=kernel, flags=flags, max_depth=5)
    try:
        ctx.render_begin(p.width, p.height)
        ctx.render_passes(np.asarray(seeds, np.int32))
        return ctx.render_read()[0]
    finally:
        ctx.render_set_params()


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_instance(cuda_ctx, ctx_no_wide, loader, monkeypatch, case):
    """Kernel 4 on layout LAY (0: shallow, top table staged; 1: the same scene with CCU_NO_TOPS; 2: embedded in a depth-13
    world) or kernel 1 on layout MODE (0: committed under CCU_NO_WIDE; 1: shallow; 2: depth 13), 3 passes of depth 5."""
    kernel, bvh, lay, i = case
    spec, nee, biome = SHADES[i]
    flags = shade_flags(spec, nee, biome)
    p = variant_scene(bvh)
    ctx = cuda_ctx
    if lay == 2:
        p = deep(p)
    if kernel == 4 and lay == 1:
        monkeypatch.setenv("CCU_NO_TOPS", "1")          # read at every launch
    if kernel == 1 and lay == 0:
        monkeypatch.setenv("CCU_NO_WIDE", "1")          # read at commit
        ctx = ctx_no_wide
    loader(ctx, p, (p.name, lay == 0 and kernel == 1))
    got = _render(ctx, p, SEEDS, kernel, flags)
    sky = staged_texels(bvh, lay == 0, spec, nee, p.sky.shape[0]) if kernel == 4 else 0
    assert ctx.last_render() == (kernel, bvh, lay, spec, nee, biome, sky)
    assert_bits(got, oracle_image(bvh, flags))


@pytest.mark.gpu
def test_reference_arrays_refuse_kernel_4(ctx_no_wide, loader, monkeypatch):
    """On a scene committed under CCU_NO_WIDE kernel 4 fails with CCU_ESTATE and launches nothing; kernel 0 picks kernel 1."""
    p = variant_scene(True)
    monkeypatch.setenv("CCU_NO_WIDE", "1")
    loader(ctx_no_wide, p, (p.name, True))
    flags = SPEC | NEE | NEAR | BIOME
    _render(ctx_no_wide, p, SEEDS[:1], 1, flags)
    before, launches = ctx_no_wide.last_render(), ctx_no_wide.launch_count()
    with pytest.raises(native.ChunkyCuError) as e:
        _render(ctx_no_wide, p, SEEDS[:1], 4, flags)
    assert e.value.code == native.CCU_ESTATE
    assert ctx_no_wide.launch_count() == launches and ctx_no_wide.last_render() == before
    got = _render(ctx_no_wide, p, SEEDS, 0, flags)
    assert ctx_no_wide.last_render() == (1, 1, 0, 1, 2, 1, 0)
    assert_bits(got, oracle_image(True, flags))


# ---------------------------------------------------------------------------------------------------------
# the selection rules (DESIGN §5), without an oracle
# ---------------------------------------------------------------------------------------------------------
FACTS = list(itertools.product((0, 1), repeat=4))     # (specular word, full-cube emitter, model emitter, biome colours)
SELECT_SKY = 16


def _fact_id(f):
    return "-".join(n if on else "no" + n for n, on in zip(("spec", "cube", "model", "biome"), f))


@functools.lru_cache(maxsize=None)
def selection_base() -> S.PackedScene:
    """A 16^3 world on a 32 x 18 canvas with both BVHs (mixed_test_scene's meshes): a stone floor with grass on top, one
    glowstone, one slab (AABB model) and one cross (quad model) on it."""
    p = S.mixed_test_scene(16, 32, 18)
    vox = np.zeros((16, 16, 16), np.int32)
    vox[:, :4, :] = S.STONE
    vox[:, 4, :] = S.GRASS
    vox[5, 5, 8], vox[8, 5, 8], vox[10, 5, 8] = S.GLOWSTONE, S.SLAB, S.CROSS
    tree, depth = S.build_octree(vox, np.arange(S.CROSS + 1, dtype=np.int64) * 2)
    return dataclasses.replace(p, octree=tree, octree_depth=depth, sky=noise_sky(SELECT_SKY, seed=3), name="select")


def selection_scene(facts) -> S.PackedScene:
    spec, cube, model, biome = facts
    p = selection_base()
    if spec:
        p = S.glossy(p)
    if not cube:
        p = dataclasses.replace(p, octree=np.where(p.octree == -2 * S.GLOWSTONE, -2 * S.STONE, p.octree).astype(np.int32))
    if model:
        p = S.emissive_models(p)
    if biome:
        p = S.with_biomes(p, seed=8, holes=0.0)
    return dataclasses.replace(p, name="select_" + _fact_id(facts))


# the 20 valid combinations of bits 4, 8, 128, 256 and 512 (128 and 256 only with 8)
SELECT_FLAGS = [s | n | b for s in (0, SPEC) for n in NEE_FLAGS for b in (0, BIOME)]


def expected_instance(facts, flags, kernel):
    """DESIGN §5 on a scene of depth 4 (layout 1, top table staged) whose BVHs the wavefront kernel can hold."""
    has_spec, has_cube, has_model, has_biome = facts
    spec = int(bool(flags & SPEC) and has_spec)
    nee = 0
    if flags & NEE:
        near = bool(flags & NEAR)
        if flags & MODELS and has_model:
            nee = 4 if near else 3
        elif has_cube:
            nee = 2 if near else 1
    biome = int(bool(flags & BIOME) and has_biome)
    bvh = int(not flags & NO_ENTITIES)
    if kernel == 1:
        return (1, bvh, 1, spec, nee, biome, 0)
    return (4, bvh, 0, spec, nee, biome, staged_texels(bvh, True, spec, nee, SELECT_SKY))


def test_selection_scenes_have_their_facts():
    for facts in FACTS:
        p = selection_scene(facts)
        assert ((p.mat_palette[5::6] != 0).any(), SO.emitter_grid(p)["has_emitters"],
                SO.emitter_grid(p, models=True)["has_emitters"], p.biome is not None) == tuple(map(bool, facts)), facts
    assert len(SELECT_FLAGS) == len(set(SELECT_FLAGS)) == 20


@pytest.mark.gpu
@pytest.mark.parametrize("facts", FACTS, ids=_fact_id)
def test_selection(cuda_ctx, loader, facts):
    """One pass on kernels 0, 1 and 4 for every valid flag set, with and without CCU_RENDER_NO_ENTITIES."""
    p = selection_scene(facts)
    loader(cuda_ctx, p, p.name)
    cuda_ctx.render_begin(p.width, p.height)
    try:
        for flags in SELECT_FLAGS:
            for f in (flags, flags | NO_ENTITIES):
                for kernel in (0, 1, 4):
                    cuda_ctx.render_set_params(kernel=kernel, flags=f)
                    cuda_ctx.render_passes(np.asarray(SEEDS[:1], np.int32))
                    assert cuda_ctx.last_render() == expected_instance(facts, f, kernel or 4), (f, kernel)
    finally:
        cuda_ctx.render_set_params()


# ---------------------------------------------------------------------------------------------------------
# sky staging at every footprint's boundary
# ---------------------------------------------------------------------------------------------------------
BOUNDARY = [(fp, r) for fp in FOOTPRINTS for r in (largest_staged_sky(fp), largest_staged_sky(fp) + 1)]


def _boundary_id(c):
    (bvh, tops, spec, nee), r = c
    return f"{'bvh' if bvh else 'nobvh'}-{'tops' if tops else 'notops'}-{'spec' if spec else 'plain'}-{'nee' if nee else 'nonee'}-sky{r}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", BOUNDARY, ids=_boundary_id)
def test_sky_staging_boundary(cuda_ctx, loader, monkeypatch, case):
    """With CCU_SKY_SMEM_MAX raised, the largest square sky that fits behind the footprint is staged and one more row is not;
    the biome kernels (the most static shared memory) with the sun off, so that every sky lookup shows."""
    (bvh, tops, spec, nee), res = case
    p = dataclasses.replace(E.without_sun(variant_scene(bvh)), sky=noise_sky(res, seed=res))
    p = dataclasses.replace(p, name=f"{p.name}_sky{res}")
    flags = BIOME | (SPEC if spec else 0) | (NEE if nee else 0)
    want = SO.FlagsOracle(p, flags).render(SEEDS)
    monkeypatch.setenv("CCU_SKY_SMEM_MAX", "1048576")
    if not tops:
        monkeypatch.setenv("CCU_NO_TOPS", "1")
    loader(cuda_ctx, p, p.name)
    got = _render(cuda_ctx, p, SEEDS, 4, flags)
    staged = res * res if res == largest_staged_sky((bvh, tops, spec, nee)) else 0
    assert cuda_ctx.last_render() == (4, bvh, 0 if tops else 1, spec, nee, 1, staged)
    assert_bits(got, want)
