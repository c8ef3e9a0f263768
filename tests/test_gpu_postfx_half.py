"""fluid_render_postfx on FLUID_FLAG_HALF_STORAGE handles: bloom, pyramid, sunrays FBOs and the mask in
dye.write are fp16 like the reference's (S:1012-1043, S:1300).  Bloom and sunrays are bit-identical to
the fp16-rounding oracle chain (postfx_half_oracle); the frame differs from it only by powf."""
import numpy as np
import pytest

from conftest import bits_equal, golden, max_rel
from postfx_half_oracle import render_postfx_half

pytestmark = pytest.mark.gpu
DT = 0.016666
POWF_TOL = 5e-6            # linearToGamma's powf: CUDA vs glibc last-place differences
# bounds against the executed-shader fixtures, measured on the CPU (test_postfx_half_cpu.py)
POW2_TARGET_TOL, RAGGED_TOL, RAGGED_TARGET_TOL = 2e-6, 1e-3, 2e-4


@pytest.fixture(scope="module")
def pkg():
    import webgl_fluid_simulation_b200 as p
    return p


def make_half(pkg, W, H, Wd, Hd, canvas=None, **cfg):
    c = {"SIM_RESOLUTION": min(W, H), "DYE_RESOLUTION": min(Wd, Hd)}
    c.update(cfg)
    cw, ch = canvas or (W, H)
    s = pkg.FluidSimulation(c, canvas_width=cw, canvas_height=ch, flags=pkg.FLAG_HALF_STORAGE, sizes=(W, H, Wd, Hd))
    assert s._dims("dye")[:2] == (Wd, Hd)
    return s


def postfx_on(s, dither, back=(10, 20, 30), **fxcfg):
    s.config.update(BLOOM=True, SUNRAYS=True, SHADING=True, BACK_COLOR={"r": back[0], "g": back[1], "b": back[2]}, **fxcfg)
    s.dithering = dither


def fp16_dye(Hd, Wd, seed):
    rng = np.random.default_rng(seed)
    dye = (rng.random((Hd, Wd, 4), dtype=np.float32) ** 4 * 3).astype(np.float32); dye[..., 3] = 1
    return dye.astype(np.float16).astype(np.float32)


@pytest.mark.parametrize("name,pow2", [("postfx_half_64_to_128", True), ("postfx_half_48x32_to_50x75", False)])
def test_half_postfx_vs_oracle_and_executed_shaders(pkg, oracle, name, pow2):
    g = golden(name)
    Wd, Hd, w, h = (int(g[k]) for k in ("Wd", "Hd", "w", "h"))
    fxcfg = dict(BLOOM_RESOLUTION=int(g["bloom_res"]), SUNRAYS_RESOLUTION=int(g["sun_res"]))
    dither = g["dither"].astype(np.float32)
    s = make_half(pkg, 16, 16, Wd, Hd)
    s.writeField("dye", g["in_dye"])
    postfx_on(s, dither, **fxcfg)
    got = s.render(w, h)
    ref = render_postfx_half(g["in_dye"], w, h, dither, cfg=fxcfg, back_rgb=(10 / 255, 20 / 255, 30 / 255))
    assert bits_equal(s.last_bloom, ref["bloom"])
    assert bits_equal(s.last_sunrays, ref["sunrays"])
    assert max_rel(got, ref["target"]) < POWF_TOL
    if pow2:
        assert bits_equal(s.last_bloom, g["bloom"]) and bits_equal(s.last_sunrays, g["sunrays"])
        assert max_rel(got, g["target"]) < POW2_TARGET_TOL
    else:
        assert max_rel(s.last_bloom, g["bloom"]) < RAGGED_TOL and max_rel(s.last_sunrays, g["sunrays"]) < RAGGED_TOL
        assert max_rel(got, g["target"]) < RAGGED_TARGET_TOL
    assert bits_equal(s.readField("dye"), g["in_dye"])        # the mask goes into dye.write only (S:1300)
    s.close()


def test_half_postfx_desktop_defaults_at_real_size(pkg, oracle):
    """The reference's desktop frame at a real size: 1280x720 canvas, DYE_RESOLUTION 576 -> 1024x576 dye,
    BLOOM_RESOLUTION 256 (455x256 bloom FBO, 8 iterations -> a 7-level pyramid), SUNRAYS_RESOLUTION 196."""
    dither = golden("postfx_half_64_to_128")["dither"].astype(np.float32)
    s = pkg.FluidSimulation({"SIM_RESOLUTION": 128, "DYE_RESOLUTION": 576}, canvas_width=1280, canvas_height=720,
                            flags=pkg.FLAG_HALF_STORAGE)
    assert s._dims("dye")[:2] == (1024, 576)
    dye = fp16_dye(576, 1024, 91)
    s.writeField("dye", dye)
    postfx_on(s, dither, BLOOM_ITERATIONS=8, BLOOM_RESOLUTION=256, SUNRAYS_RESOLUTION=196)
    got = s.render()
    assert got.shape == (720, 1280, 4)
    ref = render_postfx_half(dye, 1280, 720, dither, back_rgb=(10 / 255, 20 / 255, 30 / 255))
    assert len(ref["pyramid"]) == 7 and s.last_bloom.shape == (256, 455, 4) and s.last_sunrays.shape == (196, 348)
    assert bits_equal(s.last_bloom, ref["bloom"])
    assert bits_equal(s.last_sunrays, ref["sunrays"])
    assert max_rel(got, ref["target"]) < POWF_TOL
    assert bits_equal(s.readField("dye"), dye)
    s.close()


def test_half_postfx_transparent_backgrounds(pkg, oracle):
    """config.TRANSPARENT: checkerboard on the screen (FLUID_BACKGROUND 1) and no background, blending
    off, into a capture target (2), as on fp32 handles."""
    dither = golden("postfx_half_64_to_128")["dither"].astype(np.float32)
    Wd, Hd, w, h = 96, 64, 150, 100
    dye = fp16_dye(Hd, Wd, 92)
    s = make_half(pkg, 16, 16, Wd, Hd, canvas=(w, h))
    s.writeField("dye", dye)
    fxcfg = dict(BLOOM_RESOLUTION=64, SUNRAYS_RESOLUTION=48)
    postfx_on(s, dither, **fxcfg)
    s.config["TRANSPARENT"] = True
    for target, bg in ((False, oracle.BG_CHECKERBOARD), (True, oracle.BG_NONE)):
        got = s.render(w, h, target=target)
        ref = render_postfx_half(dye, w, h, dither, cfg=fxcfg, background=bg)
        assert bits_equal(s.last_bloom, ref["bloom"]) and bits_equal(s.last_sunrays, ref["sunrays"]), bg
        assert max_rel(got, ref["target"]) < POWF_TOL, bg
    s.close()


def test_half_postfx_short_pyramid_leaves_bloom_cleared(pkg, oracle):
    """BLOOM_ITERATIONS = 1: fewer than two pyramid levels, applyBloom returns before drawing
    (S:1353), so the bloom FBO keeps createFBO's (0,0,0,1)."""
    dither = golden("postfx_half_64_to_128")["dither"].astype(np.float32)
    dye = fp16_dye(64, 64, 93)
    s = make_half(pkg, 16, 16, 64, 64)
    s.writeField("dye", dye)
    fxcfg = dict(BLOOM_RESOLUTION=64, SUNRAYS_RESOLUTION=48, BLOOM_ITERATIONS=1)
    postfx_on(s, dither, **fxcfg)
    got = s.render(128, 128)
    assert np.all(s.last_bloom == np.array([0, 0, 0, 1], np.float32))
    ref = render_postfx_half(dye, 128, 128, dither, cfg=fxcfg, back_rgb=(10 / 255, 20 / 255, 30 / 255))
    assert bits_equal(s.last_sunrays, ref["sunrays"])
    assert max_rel(got, ref["target"]) < POWF_TOL
    s.close()


def test_half_postfx_in_the_frame_loop(pkg, oracle):
    """Splats, three steps, a post-FX frame, one more step: the frame matches the oracle on the handle's
    own dye, and the step after it is bit-identical to the half-storage oracle fed the same fields, so
    the mask left in dye.write does not leak into the simulation."""
    O = oracle
    dither = golden("postfx_half_64_to_128")["dither"].astype(np.float32)
    W, H, Wd, Hd = 64, 64, 128, 128
    s = make_half(pkg, W, H, Wd, Hd, canvas=(256, 256))
    rng = np.random.default_rng(94)
    for _ in range(4):
        x, y = rng.random(2)
        dx, dy = 1000 * (rng.random(2) - 0.5)
        s.splat(float(x), float(y), float(dx), float(dy), tuple(float(v) for v in rng.random(3) * 1.5))
    for _ in range(3):
        s.step(DT)
    fields = {n: s.readField(n) for n in ("velocity", "dye", "pressure")}
    postfx_on(s, dither)
    got = s.render()
    ref = render_postfx_half(fields["dye"], 256, 256, dither, back_rgb=(10 / 255, 20 / 255, 30 / 255))
    assert bits_equal(s.last_bloom, ref["bloom"]) and bits_equal(s.last_sunrays, ref["sunrays"])
    assert max_rel(got, ref["target"]) < POWF_TOL
    assert bits_equal(s.readField("dye"), fields["dye"])
    sim = O.OracleSim(W, H, Wd, Hd, half_storage=True)
    sim.velocity, sim.dye, sim.pressure = (fields[n].copy() for n in ("velocity", "dye", "pressure"))
    s.step(DT); sim.step(DT)
    for n in ("velocity", "dye", "pressure", "divergence", "curl"):
        assert bits_equal(s.readField(n), getattr(sim, n)), n
    s.close()
