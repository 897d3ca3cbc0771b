"""The kernels on the rays of oracle/edge_rays.py, against the CPU oracle on every pixel of every output: rays along voxel
faces and edges, from outside the cube, from inside blocks, with zero, denormal, infinite or NaN components, and the sun
at its switches.  Floats compare as "same bits, or both NaN" (the CPU's default NaN has the sign bit set, the GPU's
canonical NaN does not).  The first-hit buffers are also checked against the reference kernel's (the golden file) and,
for axis-aligned rays through voxel centres, against the geometric answer."""
import numpy as np
import pytest

from chunkyclplugin_b200.javarandom import pass_seeds
from conftest import load_scene
from oracle import edge_rays as E
from test_gpu_input_edges import _render
from test_oracle_edge_rays import E_PASSES, EDGE, SUN, assert_first_hit_matches_golden, check_axis_hits


@pytest.fixture(scope="module")
def catalogue():
    return E.scenes()


@pytest.fixture(scope="module")
def golden():
    from test_oracle_edge_rays import GOLDEN
    return np.load(GOLDEN)


@pytest.fixture(scope="module")
def ctx_no_wide():
    """A context of its own for scenes committed with CCU_NO_WIDE (the reference's arrays, layout mode 0)."""
    from chunkyclplugin_b200 import native
    ctx = native.Context(0)
    yield ctx
    ctx.close()


def assert_first_hit_equal(got, want):
    for k in ("block", "face", "node", "kind"):
        assert np.array_equal(got[k], want[k]), k
    for k in ("t", "normal", "color"):
        ok = E.same_bits_or_nan(got[k], want[k])
        assert ok.all(), (k, np.nonzero(~ok)[0][:8])


def assert_image_equal(got, want):
    ok = E.same_bits_or_nan(got, want)
    assert ok.all(), np.unique(np.nonzero(~ok)[0] // 3)[:8]


@pytest.mark.gpu
@pytest.mark.parametrize("name", EDGE)
def test_first_hit(catalogue, golden, cuda_ctx, ctx_no_wide, monkeypatch, name):
    """k_first_hit on the commit-time layouts and on the reference's arrays (CCU_NO_WIDE), against the oracle, the
    reference kernel's buffers and - on the full-cube scenes - the geometric answer."""
    import oracle
    p = catalogue[name]
    seed = pass_seeds(1)[0]
    want = oracle.Oracle(p).first_hit(seed)
    load_scene(cuda_ctx, p)
    got = cuda_ctx.first_hit(seed)
    assert_first_hit_equal(got, want)
    assert_first_hit_matches_golden(golden, name, got)
    if p.meta["base"] in E.FULL_CUBE_SCENES:
        check_axis_hits(p, got)
    monkeypatch.setenv("CCU_NO_WIDE", "1")
    load_scene(ctx_no_wide, p)
    assert_first_hit_equal(ctx_no_wide.first_hit(seed), want)


@pytest.mark.gpu
@pytest.mark.parametrize("name", EDGE)
def test_preview(catalogue, cuda_ctx, name):
    import oracle
    p = catalogue[name]
    load_scene(cuda_ctx, p)
    assert np.array_equal(cuda_ctx.preview(), oracle.Oracle(p).preview())


@pytest.mark.gpu
@pytest.mark.parametrize("sun", ["sun", "nosun"])
@pytest.mark.parametrize("name", EDGE)
def test_render(catalogue, cuda_ctx, name, sun):
    """Kernel 4 (wavefront) and kernel 1 (thread per pixel), 4 passes: the paths start on the catalogue's rays."""
    import oracle
    p = catalogue[name] if sun == "sun" else E.without_sun(catalogue[name])
    seeds = pass_seeds(E_PASSES)
    want = oracle.Oracle(p).render(seeds)
    load_scene(cuda_ctx, p)
    assert_image_equal(_render(cuda_ctx, p, seeds, 4), want)
    assert_image_equal(_render(cuda_ctx, p, seeds, 1), want)


@pytest.mark.gpu
@pytest.mark.parametrize("name", SUN)
def test_sun_at_its_switches(catalogue, cuda_ctx, name):
    """k_sun_setup's basis, through every sun sample of kernel 4 and kernel 1."""
    import oracle
    p = catalogue[name]
    seeds = pass_seeds(E_PASSES)
    want = oracle.Oracle(p).render(seeds)
    load_scene(cuda_ctx, p)
    assert_image_equal(_render(cuda_ctx, p, seeds, 4), want)
    assert_image_equal(_render(cuda_ctx, p, seeds, 1), want)
