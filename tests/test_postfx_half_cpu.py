"""Post-FX in half-float storage, CPU side: the fp16-rounding oracle chain (postfx_half_oracle) against
the executed reference shaders with half-float post-FX FBOs (tests/golden/postfx_half_*.npz, cut by
make_golden_postfx_half.py).  The GPU test's bounds against these fixtures are the ones measured here."""
import numpy as np
import pytest

from conftest import bits_equal, golden, max_rel
from postfx_half_oracle import render_postfx_half

CASES = [("postfx_half_64_to_128", True), ("postfx_half_48x32_to_50x75", False)]
# ragged grids: the rasteriser's vUv differs from (i + .5) / w in the last place and moves the LINEAR
# weights; after fp16 rounding that is at most one fp16 ulp flip (measured 5.0e-4 bloom, 3.0e-4
# sunrays, 2.4e-4 mask alpha, 5.8e-5 target)
RAGGED_TOL, RAGGED_TARGET_TOL = 1e-3, 2e-4
POW2_TARGET_TOL = 2e-6                  # pow() (linearToGamma) is implementation-defined; measured 1.7e-7


def _run(oracle_fn, g, **kw):
    return oracle_fn(g["in_dye"], int(g["w"]), int(g["h"]), g["dither"].astype(np.float32),
                     cfg=dict(BLOOM_RESOLUTION=int(g["bloom_res"]), SUNRAYS_RESOLUTION=int(g["sun_res"])),
                     back_rgb=tuple(float(x) / 255 for x in g["back"]), **kw)


@pytest.mark.parametrize("name,pow2", CASES)
def test_half_chain_matches_executed_shaders_with_half_fbos(oracle, name, pow2):
    g = golden(name)
    r = _run(render_postfx_half, g)
    n = len([k for k in g.files if k.startswith("pyr")])
    assert n >= 2 and len(r["pyramid"]) == n
    if pow2:
        assert bits_equal(r["bloom"], g["bloom"]) and bits_equal(r["sunrays"], g["sunrays"])
        assert bits_equal(r["mask_alpha"], g["mask_alpha"])
        assert all(bits_equal(r["pyramid"][k], g[f"pyr{k}"]) for k in range(n))
        assert max_rel(r["target"], g["target"]) < POW2_TARGET_TOL
    else:
        for k in ("bloom", "sunrays", "mask_alpha"):
            assert max_rel(r[k], g[k]) < RAGGED_TOL, k
        assert max_rel(r["target"], g["target"]) < RAGGED_TARGET_TOL


@pytest.mark.parametrize("name,pow2", CASES)
def test_half_fixtures_hold_fp16_values(name, pow2):
    """Every post-FX FBO of the fixtures is a half-float texture, and so is the input dye."""
    g = golden(name)
    keys = ["in_dye", "bloom", "sunrays", "mask_alpha"] + [k for k in g.files if k.startswith("pyr")]
    for k in keys:
        a = np.ascontiguousarray(g[k], np.float32)
        assert bits_equal(a, a.astype(np.float16).astype(np.float32)), k


@pytest.mark.parametrize("name,pow2", CASES)
def test_fp32_chain_is_not_the_half_chain(oracle, name, pow2):
    """The fixtures discriminate: widening the fp16 dye and running the fp32-FBO chain lands more
    than 1e-4 away from the half-float reference (4e-4 to 7e-4 measured)."""
    g = golden(name)
    r = _run(oracle.render_postfx, g)
    for k in ("bloom", "sunrays", "target"):
        assert not bits_equal(r[k], g[k]), k
        assert max_rel(r[k], g[k]) > 1e-4, k


def test_half_chain_rounds_every_fbo_and_keeps_the_target_fp32(oracle):
    """Structure of the chain on a small input: every FBO it returns is fp16-valued, the target is not,
    and with fewer than two pyramid levels applyBloom returns early, leaving the bloom FBO at its
    (0,0,0,1) clear."""
    rng = np.random.default_rng(5)
    dye = oracle.round_half((rng.random((20, 30, 4), dtype=np.float32) ** 2 * 2).astype(np.float32))
    dither = rng.random((8, 8, 3), dtype=np.float32)
    r = render_postfx_half(dye, 45, 33, dither, cfg=dict(BLOOM_RESOLUTION=32, SUNRAYS_RESOLUTION=24))
    for a in [r["bloom"], r["sunrays"], r["mask"]] + r["pyramid"]:
        assert bits_equal(a, oracle.round_half(a))
    assert not bits_equal(r["target"], oracle.round_half(r["target"]))
    r = render_postfx_half(dye, 45, 33, dither, cfg=dict(BLOOM_RESOLUTION=32, SUNRAYS_RESOLUTION=24, BLOOM_ITERATIONS=1))
    assert r["pyramid"] == [] and np.all(r["bloom"] == np.array([0, 0, 0, 1], np.float32))
