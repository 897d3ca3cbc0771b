"""North-star acceptance checks at the BASELINE configurations' real sizes (BASELINE.json configs 1-5).

(a) CUDA (through the C ABI) vs the reference's UNMODIFIED OpenCL kernel, strict build (IEEE arithmetic: the
    contract of DESIGN.md section 2), on the full frame: hit flag / block id / face bit-exact, distance and
    normal bit-exact.  Reference entry point: closestIntersect (K/kernel.h:14-24) called for the camera rays of
    K/rayTracer.cl:55-91.
(b) CUDA vs the stock build (what a Chunky user runs): converged radiance, per-pixel RMSE / mean <= 1 % over a strided
    pixel sample, full-frame image means within 0.2 %.
    For the dark indoor scene (config 3) the difference is Monte-Carlo noise of paths that take another branch at
    a knife edge; that claim is tested: a second reference run on a DISJOINT seed stream at the same spp gives
    the noise floor, and rmse(ours, ref) must stay below it.
(c) CUDA vs the C oracle, bit-exact, on a strided pixel subset of every BASELINE config at its real size
    (the oracle restates K/rayTracer.cl:11-113 on the CPU; tests/test_oracle_golden.py pins it to the reference).

(a)/(b) compare with outputs of the reference kernel stored in tests/golden/acceptance_reference.npz (oracle/golden.py
says what it holds; scripts/acceptance_golden.py produced it on a B200).
"""
import numpy as np
import pytest

from chunkyclplugin_b200.javarandom import pass_seeds
from conftest import load_scene
from oracle import golden

pytestmark = pytest.mark.gpu


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


@pytest.fixture(scope="module")
def full_scenes():
    """BASELINE configs at their real sizes (built once per module)."""
    from chunkyclplugin_b200 import scenes as S
    cache = {}

    def get(name):
        if name not in cache:
            if name == "config1":
                cache[name] = S.terrain_scene(256, 1920, 1080)
            elif name == "config3":
                cache[name] = S.indoor_scene(256, 1920, 1080)
            elif name == "config4":
                cache[name] = S.entity_scene(256, 1920, 1080)
            elif name == "config5":
                cache[name] = S.large_world_scene(width=3840, height=2160)
            else:
                raise KeyError(name)
        return cache[name]
    return get


@pytest.fixture(scope="module")
def reference():
    return np.load(golden.PATH)


def _face_of(normal):
    n = normal.reshape(-1, 3)
    face = np.full(n.shape[0], 6, np.int32)
    for f, v in enumerate([(-1, 0, 0), (1, 0, 0), (0, -1, 0), (0, 1, 0), (0, 0, -1), (0, 0, 1)]):
        face[(n == np.array(v, np.float32)).all(axis=1)] = f
    return face


# ---------------------------------------------------------------------------------------------------------
# (a) first-hit buffers, full frame, vs the strict build of the reference kernel
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("config", ["config1", "config3", "config4", "config5"])
def test_first_hit_full_frame_vs_reference_kernel(config, full_scenes, reference, cuda_ctx):
    p = full_scenes(config)
    load_scene(cuda_ctx, p)
    got = cuda_ctx.first_hit(pass_seeds(1)[0])
    hit = got["kind"] > 0
    n = hit.size
    assert n == p.width * p.height
    assert hit.any()
    # the sampled pixels first, so that a difference is reported where it is
    idx = golden.sample_pixels(n, golden.FIRST_HIT_SAMPLES)
    w = {k: reference[f"fh_{config}_{k}"] for k in ("hit", "block", "t", "normal", "color")}
    sh = w["hit"] != 0
    assert np.array_equal(hit[idx], sh), f"{config}: hit flag differs in {(hit[idx] != sh).sum()} of {idx.size} sampled pixels"
    # octree hits: record.material is the block id; BVH hits keep the stale octree value there (SURVEY Q15) - compare as the reference reports it
    assert np.array_equal(got["block"][idx][sh], w["block"][sh]), f"{config}: block id differs in sampled hit pixels"
    assert np.array_equal(_bits(got["t"][idx][sh]), _bits(w["t"][sh])), f"{config}: hit distance not bit-exact"
    assert np.array_equal(_bits(got["normal"].reshape(-1, 3)[idx][sh]), _bits(w["normal"][sh])), f"{config}: normal not bit-exact"
    assert np.array_equal(got["face"][idx][sh], _face_of(w["normal"])[sh]), f"{config}: face differs"
    assert np.array_equal(_bits(got["color"].reshape(-1, 4)[idx][sh]), _bits(w["color"][sh])), f"{config}: surface colour not bit-exact"
    # the full frame, bit for bit
    assert np.array_equal(got["face"][hit], _face_of(got["normal"])[hit]), f"{config}: face disagrees with the normal"
    digests = golden.first_hit_digests(hit, got["block"], got["t"], got["normal"], got["color"])
    for k, v in digests.items():
        assert v == str(reference[f"fh_{config}_digest_{k}"]), f"{config}: full-frame {k} differs from the reference kernel's"


# ---------------------------------------------------------------------------------------------------------
# (b) converged radiance vs the stock build
# ---------------------------------------------------------------------------------------------------------
def _rel_rmse(a, b):
    a = a.astype(np.float64)
    b = b.astype(np.float64)
    return float(np.sqrt(np.mean((a - b) ** 2)) / b.mean())


def _ours(ctx, p, seeds):
    ctx.render_begin(p.width, p.height)
    ctx.render_passes(np.asarray(seeds, np.int32))
    img, spp = ctx.render_read()
    assert spp == len(seeds)
    return img


@pytest.mark.parametrize("config,spp", [("config1", 256), ("config4", 64)])
def test_converged_radiance_vs_reference_kernel(config, spp, full_scenes, reference, cuda_ctx):
    p = full_scenes(config)
    load_scene(cuda_ctx, p)
    got = _ours(cuda_ctx, p, pass_seeds(spp))
    want = reference[f"rad_{config}_rgb"]
    rel = _rel_rmse(got.reshape(-1, 3)[golden.sample_pixels(p.width * p.height, golden.RADIANCE_SAMPLES)], want)
    assert np.isfinite(got).all()
    assert rel <= 0.01, f"{config}: RMSE / mean = {rel:.4%} at {spp} spp (north-star bound 1 %)"
    assert abs(float(got.mean()) / float(reference[f"rad_{config}_mean"]) - 1.0) < 2e-3


def test_converged_radiance_indoor_with_noise_floor(full_scenes, reference, cuda_ctx):
    """Config 3 at its BASELINE 1024 spp: rmse(ours, ref) against the reference's own seed-to-seed noise (a second
    reference run on the disjoint seed stream of JavaRandom(987654321), same spp, same sampled pixels)."""
    p = full_scenes("config3")
    load_scene(cuda_ctx, p)
    got = _ours(cuda_ctx, p, pass_seeds(1024))
    want = reference["rad_config3_rgb"]
    rel = _rel_rmse(got.reshape(-1, 3)[golden.sample_pixels(p.width * p.height, golden.RADIANCE_SAMPLES)], want)
    floor = float(reference["rad_config3_noise_floor"])
    assert np.isfinite(got).all()
    # same seeds: only the paths that branch differently at a knife edge differ, so we must sit well inside the noise floor
    assert rel <= 1.1 * floor, f"ours vs ref {rel:.4%} exceeds the reference's own seed-to-seed noise {floor:.4%}"
    assert rel <= 0.01 or rel <= 0.5 * floor, f"RMSE / mean = {rel:.4%} (bound 1 %, noise floor {floor:.4%})"
    assert abs(float(got.mean()) / float(reference["rad_config3_mean"]) - 1.0) < 2e-3


# ---------------------------------------------------------------------------------------------------------
# (c) CUDA vs oracle, bit-exact, strided pixels of every BASELINE config at its real size
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("config,passes", [("config1", 8), ("config3", 8), ("config4", 4), ("config5", 4)])
def test_render_strided_vs_oracle_at_full_size(config, passes, full_scenes, cuda_ctx):
    import oracle
    p = full_scenes(config)
    load_scene(cuda_ctx, p)
    seeds = pass_seeds(passes)
    got = _ours(cuda_ctx, p, seeds).reshape(-1, 3)
    gids = np.arange(17, p.width * p.height, 64, dtype=np.int32)
    ref = oracle.Oracle(p).render(seeds, gids=gids).reshape(-1, 3)
    bad = (_bits(got[gids]) != _bits(ref[gids])).any(axis=1)
    assert not bad.any(), f"{config}: {bad.sum()} of {gids.size} sampled pixels differ from the oracle"
    assert got[gids].max() > 0


@pytest.mark.parametrize("config", ["config1", "config5"])
def test_first_hit_vs_oracle_at_full_size(config, full_scenes, cuda_ctx):
    """Config 2 (first-hit pass) incl. the octree node index, which the reference kernel has no output for."""
    import oracle
    p = full_scenes(config)
    load_scene(cuda_ctx, p)
    seed = pass_seeds(1)[0]
    got = cuda_ctx.first_hit(seed)
    ref = oracle.Oracle(p).first_hit(seed)
    for k in ("block", "face", "node", "kind"):
        assert np.array_equal(got[k], ref[k]), f"{config}: {k} differs in {(got[k] != ref[k]).sum()} pixels"
    for k in ("t", "normal", "color"):
        assert np.array_equal(_bits(got[k]), _bits(ref[k])), f"{config}: {k} differs"
