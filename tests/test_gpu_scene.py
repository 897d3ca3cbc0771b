"""Re-commit, partial update, render flags and replication of a committed scene: each must render, bit for bit, as a fresh
context that loaded the final scene once (thread-per-pixel and wavefront kernels, first-hit buffers and preview)."""
import dataclasses

import numpy as np
import pytest

from chunkyclplugin_b200 import scenes as S
from chunkyclplugin_b200.javarandom import pass_seeds
from conftest import load_scene

pytestmark = pytest.mark.gpu

SEEDS = pass_seeds(4)


def _outputs(ctx, p, flags=0):
    """Every output a committed scene feeds, as raw bytes (the camera is set)."""
    out = {}
    for kernel in (4, 1):
        ctx.render_set_params(kernel=kernel, flags=flags)
        ctx.render_begin(p.width, p.height)
        ctx.render_passes(SEEDS)
        img, spp = ctx.render_read()
        assert spp == len(SEEDS)
        out[f"kernel{kernel}"] = img.copy()
    out.update({f"first_hit_{k}": v for k, v in ctx.first_hit(77).items()})
    out["preview"] = ctx.preview()
    ctx.render_end()
    return {k: v.view(np.uint8) for k, v in out.items()}


def _fresh(p, flags=0, device=0):
    from chunkyclplugin_b200 import native
    with native.Context(device) as ctx:
        load_scene(ctx, p)
        return _outputs(ctx, p, flags), ctx.scene_device_bytes()


def _assert_same(got, want):
    assert got.keys() == want.keys()
    for k in want:
        assert np.array_equal(got[k], want[k]), k


def _new_sun(p):
    return S.pack_sun(int(p.sun[1]), int(p.sun[2]), intensity=2.0, altitude=0.6, azimuth=2.4)


@pytest.mark.parametrize("name", ["terrain64", "entities"])
def test_second_commit_of_an_unchanged_scene(scenes, name):
    from chunkyclplugin_b200 import native
    p = scenes(name)
    want, want_bytes = _fresh(p)
    with native.Context(0) as ctx:
        load_scene(ctx, p)
        ctx.scene_commit()
        assert ctx.scene_device_bytes() == want_bytes
        _assert_same(_outputs(ctx, p), want)


@pytest.mark.parametrize("name,setter", [("terrain64", "set_sun"), ("entities", "set_world_bvh")])
def test_one_setter_then_commit_without_scene_begin(scenes, name, setter):
    from chunkyclplugin_b200 import native
    p = scenes(name)
    field, value = ("sun", _new_sun(p)) if setter == "set_sun" else ("world_bvh", S.EMPTY_BVH.copy())
    final = dataclasses.replace(p, **{field: value})
    want, want_bytes = _fresh(final)
    assert not np.array_equal(want["kernel1"], _fresh(p)[0]["kernel1"])   # the update changes the image
    with native.Context(0) as ctx:
        load_scene(ctx, p)
        ctx.render_passes(SEEDS)
        getattr(ctx, setter)(value)
        with pytest.raises(native.ChunkyCuError) as err:
            ctx.render_passes(SEEDS)
        assert err.value.code == native.CCU_ESTATE
        ctx.scene_commit()
        assert ctx.scene_device_bytes() == want_bytes
        _assert_same(_outputs(ctx, final), want)


def test_no_entities_flag_on_and_off(scenes):
    from chunkyclplugin_b200 import native
    p = scenes("entities")
    want_on, _ = _fresh(p, flags=native.CCU_RENDER_NO_ENTITIES)
    want_off, _ = _fresh(p)
    assert not np.array_equal(want_on["kernel1"], want_off["kernel1"])
    with native.Context(0) as ctx:
        load_scene(ctx, p)
        _assert_same(_outputs(ctx, p, flags=native.CCU_RENDER_NO_ENTITIES), want_on)
        _assert_same(_outputs(ctx, p), want_off)


def test_replica_committed_again_with_a_new_sun(scenes):
    from chunkyclplugin_b200 import native
    if native.device_count() < 2:
        pytest.skip("NEEDS 2 GPUs - replication is not exercised on this box")
    p = scenes("entities")
    final = dataclasses.replace(p, sun=_new_sun(p))
    want, _ = _fresh(final, device=1)
    group = native.Group(devices=[0, 1])
    try:
        m0, m1 = group.member(0), group.member(1)
        load_scene(m0, p)
        m0.render_end()
        group.replicate_scene()
        assert m1.scene_device_bytes() == m0.scene_device_bytes()
        m1.set_sun(final.sun)
        m1.scene_commit()
        m1.camera_set(p.projector_type, p.camera)
        _assert_same(_outputs(m1, final), want)
    finally:
        group.close()
