"""Teardown with work in flight, and a second scene loaded into a used context: what follows must render exactly as a context
that never saw the earlier work."""
import numpy as np
import pytest

from chunkyclplugin_b200.javarandom import pass_seeds
from conftest import load_scene

pytestmark = pytest.mark.gpu


def _merged(p, seeds):
    """A fresh context renders `seeds` as one window and merges it into a zeroed sample buffer."""
    from chunkyclplugin_b200 import native
    with native.Context(0) as ctx:
        load_scene(ctx, p)
        sb = np.zeros(p.width * p.height * 3, dtype=np.float64)
        ctx.render_passes(seeds)
        assert ctx.render_merge(sb, 0) == len(seeds)
        ctx.render_end()
    return sb


def _load_group_scene(group, p):
    load_scene(group.member(0), p)
    group.member(0).render_end()
    group.camera_set(p.projector_type, p.camera)
    group.render_begin(p.width, p.height)


def _group_merged(p, seeds):
    from chunkyclplugin_b200 import native
    group = native.Group(devices=[0])
    try:
        _load_group_scene(group, p)
        sb = np.zeros(p.width * p.height * 3, dtype=np.float64)
        group.render_passes(seeds)
        assert group.render_merge(sb, 0) == len(seeds)
        group.render_end()
    finally:
        group.close()
    return sb


def test_context_destroyed_with_passes_queued_and_merge_running(scenes):
    from chunkyclplugin_b200 import native
    p = scenes("terrain64")
    seeds = pass_seeds(64)
    want = _merged(p, seeds)
    ctx = native.Context(0)
    load_scene(ctx, p)
    sb = np.zeros(p.width * p.height * 3, dtype=np.float64)
    ctx.render_passes(seeds[:16], block=False)
    assert ctx.render_merge_async(sb, 0) == 16       # the merge worker waits for the read-back of this window ...
    ctx.render_passes(pass_seeds(512), block=False)  # ... while the next window is queued behind it
    ctx.close()
    assert np.array_equal(_merged(p, seeds), want)


def test_group_destroyed_right_after_async_merge(scenes):
    from chunkyclplugin_b200 import native
    p = scenes("terrain64")
    seeds = pass_seeds(24)
    want = _group_merged(p, seeds)
    group = native.Group(devices=[0])
    _load_group_scene(group, p)
    sb = np.zeros(p.width * p.height * 3, dtype=np.float64)
    group.render_passes(seeds)
    assert group.render_merge_async(sb, 0) == len(seeds)
    group.close()                                    # no render_merge_wait: the destroy joins the merge
    assert np.array_equal(_group_merged(p, seeds), want)


def test_second_scene_replaces_the_first(scenes):
    """Scene A (entity BVHs, models, triangles) then scene B in one context == a fresh context that only loaded B."""
    from chunkyclplugin_b200 import native
    a, b = scenes("entities"), scenes("terrain64")
    seeds = pass_seeds(8)

    def render(ctx):
        ctx.render_passes(seeds)
        img, spp = ctx.render_read()
        assert spp == len(seeds)
        ctx.render_end()
        return img, ctx.scene_device_bytes()

    with native.Context(0) as fresh:
        load_scene(fresh, b)
        want_img, want_bytes = render(fresh)
    with native.Context(0) as ctx:
        load_scene(ctx, a)
        render(ctx)
        load_scene(ctx, b)
        img, nbytes = render(ctx)
    assert nbytes == want_bytes
    assert np.array_equal(img.view(np.uint32), want_img.view(np.uint32))
