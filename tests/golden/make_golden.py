"""Cuts tests/golden/*.npz by EXECUTING the reference's GLSL shader text (oracle/glsl_exec.py).

Run in the build container only (needs /root/reference/script.js):
    python tests/golden/make_golden.py
    python tests/golden/make_golden.py citations    # script_js_citations.json only
The .npz files are committed; the tests never read /root/reference.
Inputs are seeded; every file stores inputs and the reference-shader outputs, fp32 storage,
`!supportLinearFiltering` path (MANUAL_FILTERING + NEAREST samplers: arithmetic fully defined by the
shader text).  `p4_*` files additionally hold the fp16-storage / LINEAR-sampler variants that the
reference uses on a desktop GPU; they are REPORT-ONLY (see DESIGN.md "Parity").
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import glsl_exec as G  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
DT = np.float32(0.016666)  # the calcDeltaTime clamp, S:1191


def mulberry32(seed):
    """Deterministic stand-in for Math.random() (the reference is unseeded, S:1433-1436)."""
    state = [seed & 0xFFFFFFFF]

    def rnd():
        state[0] = (state[0] + 0x6D2B79F5) & 0xFFFFFFFF
        t = state[0]
        t = ((t ^ (t >> 15)) * (t | 1)) & 0xFFFFFFFF
        t ^= (t + (((t ^ (t >> 7)) * (t | 61)) & 0xFFFFFFFF)) & 0xFFFFFFFF
        return ((t ^ (t >> 14)) & 0xFFFFFFFF) / 4294967296.0
    return rnd


def hsv_to_rgb(h, s, v):                     # HSVtoRGB S:1573-1597
    i = int(np.floor(h * 6)); f = h * 6 - i
    p = v * (1 - s); q = v * (1 - f * s); t = v * (1 - (1 - f) * s)
    return [(v, t, p), (q, v, p), (p, v, t), (p, q, v), (t, p, v), (v, p, q)][i % 6]


def splat_list(n, seed):
    """multipleSplats(n) argument stream, S:1427-1439 (+ generateColor S:1565-1571)."""
    rnd = mulberry32(seed); out = []
    for _ in range(n):
        r, g, b = hsv_to_rgb(rnd(), 1.0, 1.0)
        col = (r * 0.15 * 10.0, g * 0.15 * 10.0, b * 0.15 * 10.0)
        x, y = rnd(), rnd()
        dx, dy = 1000 * (rnd() - 0.5), 1000 * (rnd() - 0.5)
        out.append((x, y, dx, dy) + col)
    return np.array(out, np.float32)


def per_pass(W, H, Wd, Hd, seed):
    rng = np.random.default_rng(seed)
    s = G.GLSLSim(W, H, Wd, Hd)
    v = (rng.standard_normal((H, W, 2)) * 50).astype(np.float32)
    dye = rng.random((Hd, Wd, 4), dtype=np.float32)
    p = rng.standard_normal((H, W)).astype(np.float32)
    s.load(velocity=v, dye=dye, pressure=p)
    o = dict(W=W, H=H, Wd=Wd, Hd=Hd, dt=DT, in_velocity=v, in_dye=dye, in_pressure=p)
    s.run_curl(); o["curl"] = s.fields()["curl"]
    s.run_vorticity(DT); o["vorticity"] = s.fields()["velocity"]
    s.run_divergence(); o["divergence"] = s.fields()["divergence"]
    s.run_clear(); o["clear"] = s.fields()["pressure"]
    s.run_pressure(1); o["jacobi1"] = s.fields()["pressure"]
    s.run_pressure(12); o["jacobi13"] = s.fields()["pressure"]
    s.run_gradient_subtract(); o["gradient"] = s.fields()["velocity"]
    s.run_advect_velocity(DT); o["advect_velocity"] = s.fields()["velocity"]
    s.run_advect_dye(DT); o["advect_dye"] = s.fields()["dye"]
    sp = np.array([0.3, 0.6, 123.0, -456.0, 0.5, 0.2, 0.9], np.float32)
    s.splat(*sp[:4], tuple(sp[4:])); f = s.fields()
    o["splat_args"] = sp; o["splat_velocity"] = f["velocity"]; o["splat_dye"] = f["dye"]
    np.savez_compressed(os.path.join(OUT, f"pass_{W}x{H}_{Wd}x{Hd}.npz"), **o)


def scenario(name, W, H, Wd, Hd, nsplat, steps, config, seed, **kw):
    s = G.GLSLSim(W, H, Wd, Hd, config=config, **kw)
    sp = splat_list(nsplat, seed)
    for a in sp:
        s.splat(*a[:4], tuple(a[4:]))
    o = dict(W=W, H=H, Wd=Wd, Hd=Hd, dt=DT, splats=sp, steps=steps,
             config_keys=np.array(list(config.keys())), config_vals=np.array(list(config.values()), np.float32))
    f = s.fields(); o["init_velocity"] = f["velocity"]; o["init_dye"] = f["dye"]
    for k in range(steps):
        s.step(DT)
        f = s.fields()
        if k + 1 in (1, 2, steps):
            for n, a in f.items():
                o[f"s{k+1}_{n}"] = a
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **o)


def display(name, Wd, Hd, w, h, seed):
    """render() with bloom / sunrays off: executed colorShader + displayShaderSource, blended."""
    rng = np.random.default_rng(seed)
    s = G.GLSLSim(16, 16, Wd, Hd)
    dye = (rng.random((Hd, Wd, 4), dtype=np.float32) * 2).astype(np.float32); dye[..., 3] = 1
    s.load(dye=dye)
    o = dict(Wd=Wd, Hd=Hd, w=w, h=h, in_dye=dye, back=np.array([30, 60, 200], np.float32))
    o["shaded"] = s.render(w, h, True, (30, 60, 200))
    o["flat"] = s.render(w, h, False, (30, 60, 200))
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **o)


def postfx(name, Wd, Hd, w, h, seed, bloom_res=64, sun_res=48):
    """render(null) with SHADING + BLOOM + SUNRAYS: the executed bloom / sunrays / blur / display
    shaders with the reference's FBO pyramid and blending.  The dithering texture is decoded from
    the reference's LDR_LLL1_0.png here and stored in the fixture (row 0 = first image row)."""
    from PIL import Image
    dither = np.asarray(Image.open("/root/reference/LDR_LLL1_0.png").convert("RGB"), dtype=np.float32) / np.float32(255.0)
    rng = np.random.default_rng(seed)
    s = G.GLSLSim(16, 16, Wd, Hd)
    dye = (rng.random((Hd, Wd, 4), dtype=np.float32) ** 4 * 3).astype(np.float32); dye[..., 3] = 1
    s.load(dye=dye)
    # small FBOs keep the fixture small; the chain (prefilter, pyramid down / additive up, final,
    # mask, march, blur, display) is the same as with the 256 / 196 defaults
    r = s.render_postfx(w, h, dither, cfg=dict(BLOOM_RESOLUTION=bloom_res, SUNRAYS_RESOLUTION=sun_res), back_color=(10, 20, 30))
    o = dict(Wd=Wd, Hd=Hd, w=w, h=h, bloom_res=bloom_res, sun_res=sun_res, in_dye=dye, dither=dither.astype(np.float16), back=np.array([10, 20, 30], np.float32),
             target=r["target"], bloom=r["bloom"].astype(np.float32), sunrays=r["sunrays"], mask_alpha=r["mask_alpha"])
    for k, t in enumerate(r["pyramid"]):
        o[f"pyr{k}"] = t
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **o)


def resample(name, Ws, Hs, Wd, Hd, ch, seed):
    """resizeFBO (S:1108-1114): the executed copyShader (S:496-506) drawn into a new Wd x Hd FBO
    while sampling the old Ws x Hs texture through its LINEAR filter (`filtering` of S:988 on the
    default desktop path; the NEAREST variant is stored too for reference)."""
    js = open(G.REFERENCE_JS).read()
    rng = np.random.default_rng(seed)
    src = (rng.standard_normal((Hs, Ws, ch)) * 3).astype(np.float32)
    o = dict(Ws=Ws, Hs=Hs, Wd=Wd, Hd=Hd, ch=ch, src=src)
    for tag, lin in (("linear", True), ("nearest", False)):
        old = G.Texture(Ws, Hs, ch, lin)
        old.store(G.V(np.concatenate([src, np.zeros((Hs, Ws, 4 - ch), np.float32)], axis=-1)))
        new = G.Texture(Wd, Hd, ch, lin)
        prog = G.Program(js, "baseVertexShader", "copyShader")
        prog.set(uTexture=old, texelSize=(0.0, 0.0))   # copyProgram never sets texelSize (S:1111): default 0
        prog.blit(new)
        o[tag] = new.data[..., :ch].copy()
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **o)


def citations():
    """script_js_citations.json for tests/test_citations_and_plan.py: the line count of script.js and
    the 1-based lines on which each of that test's spot-check needles occurs (no script.js text)."""
    import json
    sys.path.insert(0, os.path.dirname(OUT))
    from test_citations_and_plan import SPOT_CHECKS
    js = open(G.REFERENCE_JS).read().splitlines()
    needles = sorted({needle for _, _, needle in SPOT_CHECKS})
    ref = {"lines": len(js), "needle_lines": {s: [k + 1 for k, l in enumerate(js) if s in l] for s in needles}}
    with open(os.path.join(OUT, "script_js_citations.json"), "w") as f:
        json.dump(ref, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "citations":
        citations()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "r02":     # the vectors added in round 2 only
        resample("resample_v_32_to_48", 32, 32, 48, 48, 2, 31)           # up-sample, ragged ratio
        resample("resample_dye_64_to_32", 64, 64, 32, 32, 4, 32)         # down-sample by 2 (power of two)
        resample("resample_dye_40x28_to_64x48", 40, 28, 64, 48, 4, 33)
        # TRANSPARENT: checkerboard under the display on the screen, bare display into a capture target
        rng = np.random.default_rng(41)
        gs = G.GLSLSim(16, 16, 64, 32)
        dye = (rng.random((32, 64, 4), dtype=np.float32) ** 3 * 1.5).astype(np.float32); dye[..., 3] = 1
        gs.load(dye=dye)
        np.savez_compressed(os.path.join(OUT, "display_transparent_64x32_to_128x64.npz"), in_dye=dye, w=128, h=64,
                            checker=gs.render(128, 64, True, transparent=True, to_screen=True),
                            bare=gs.render(128, 64, True, transparent=True, to_screen=False))
        # BASELINE configs[0]: 128x128 sim / 256x256 dye, 20 iterations (the reference's own defaults
        # except the dye size) -- two whole steps after multipleSplats(5)
        scenario("config0_128_256", 128, 128, 256, 256, 5, 2, dict(CURL=30, PRESSURE_ITERATIONS=20), 4321)
        print("round-2 golden vectors written to", OUT)
        sys.exit(0)
    postfx("postfx_64_to_128", 64, 64, 128, 128, 21)           # power-of-two target, dye and bloom FBO
    postfx("postfx_48x32_to_50x75", 48, 32, 50, 75, 22)        # ragged, portrait canvas
    display("display_64_to_128", 64, 64, 128, 128, 11)      # power-of-two target: bitwise
    display("display_40x28_to_50x30", 40, 28, 50, 30, 12)   # ragged: vUv rounding -> tolerance
    per_pass(32, 32, 64, 64, 1)
    per_pass(24, 16, 40, 28, 2)      # non-square, non-power-of-two, Wd/W not integer
    per_pass(64, 32, 128, 64, 3)
    per_pass(16, 16, 16, 16, 4)      # dye at sim resolution (BASELINE configs 3-5)
    scenario("step_curl30_32", 32, 32, 64, 64, 8, 3, dict(CURL=30, PRESSURE_ITERATIONS=20), 1234)
    scenario("step_curl0_32", 32, 32, 64, 64, 8, 20, dict(CURL=0, PRESSURE_ITERATIONS=20), 1234)
    scenario("step_curl30_48x32", 48, 32, 96, 64, 6, 2, dict(CURL=30, PRESSURE_ITERATIONS=7), 99)
    # report-only: what a desktop browser actually runs (LINEAR samplers + half-float textures)
    scenario("p4_linear_half_32", 32, 32, 64, 64, 8, 3, dict(CURL=30, PRESSURE_ITERATIONS=20), 1234,
             linear_filtering=True, half=True)
    scenario("p4_linear_fp32_32", 32, 32, 64, 64, 8, 3, dict(CURL=30, PRESSURE_ITERATIONS=20), 1234,
             linear_filtering=True, half=False)
    print("golden vectors written to", OUT)
