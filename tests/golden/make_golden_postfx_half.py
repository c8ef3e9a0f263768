"""Cuts tests/golden/postfx_half_*.npz: render(null) with SHADING + BLOOM + SUNRAYS by EXECUTING the
reference's GLSL shader text (oracle/glsl_exec.py) with the texture formats a desktop browser uses,
i.e. half-float storage.

Run in the build container only (needs the reference's script.js and LDR_LLL1_0.png):
    python tests/golden/make_golden_postfx_half.py
It writes postfx_half_64_to_128.npz and postfx_half_48x32_to_50x75.npz and nothing else.  Shapes,
seeds, FBO sizes and back colour are those of postfx_64_to_128 / postfx_48x32_to_50x75
(make_golden.py postfx()), with the input dye rounded to fp16 (the RGBA16F dye texture, S:986-1006).
The bloom FBO, the pyramid, the sunrays mask (drawn into dye.write, RGBA16F: S:1300) and both sunrays
FBOs are half-float textures (S:1012-1043): every blit into them rounds its output to fp16, the
additive up-sampling blend included.  The final target is fp32.  The keys are those of the fp32
post-FX fixtures.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import glsl_exec as G  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
F = np.float32


def executed_postfx_half(dye_arr, width, height, dither, cfg, back_color):
    """GLSLSim.render_postfx's blit sequence (applyBloom S:1350-1394, applySunrays + blur S:1396-1419,
    drawColor + drawDisplay S:1296-1348) with half=True on every post-FX FBO."""
    js = open(G.REFERENCE_JS).read()
    c = dict(BLOOM_ITERATIONS=8, BLOOM_RESOLUTION=256, BLOOM_INTENSITY=0.8, BLOOM_THRESHOLD=0.6,
             BLOOM_SOFT_KNEE=0.7, SUNRAYS_RESOLUTION=196, SUNRAYS_WEIGHT=1.0)
    c.update(cfg)

    def get_resolution(res):                                                    # S:1612-1624
        ar = width / height
        if ar < 1: ar = 1.0 / ar
        mn, mx = int(np.floor(res + 0.5)), int(np.floor(res * ar + 0.5))
        return (mx, mn) if width > height else (mn, mx)

    P = lambda vs, fs, d=(): G.Program(js, vs, fs, d)
    dye = G.Texture(dye_arr.shape[1], dye_arr.shape[0], 4, True, half=True); dye.data = dye_arr.copy()
    bw, bh = get_resolution(c["BLOOM_RESOLUTION"])
    bloom = G.Texture(bw, bh, 4, True, half=True)
    pyramid = []
    for i in range(c["BLOOM_ITERATIONS"]):
        pw, ph = bw >> (i + 1), bh >> (i + 1)
        if pw < 2 or ph < 2: break
        pyramid.append(G.Texture(pw, ph, 4, True, half=True))
    if len(pyramid) >= 2:
        knee = c["BLOOM_THRESHOLD"] * c["BLOOM_SOFT_KNEE"] + 0.0001
        pre = P("baseVertexShader", "bloomPrefilterShader")
        pre.set(texelSize=(0.0, 0.0), curve=(c["BLOOM_THRESHOLD"] - knee, knee * 2, 0.25 / knee),
                threshold=c["BLOOM_THRESHOLD"], uTexture=dye)
        pre.blit(bloom)
        last = bloom
        blurp = P("baseVertexShader", "bloomBlurShader")
        for dest in pyramid:
            blurp.set(texelSize=(last.texelSizeX, last.texelSizeY), uTexture=last)
            blurp.blit(dest); last = dest
        for i in range(len(pyramid) - 2, -1, -1):
            base = pyramid[i]
            blurp.set(texelSize=(last.texelSizeX, last.texelSizeY), uTexture=last)
            blurp.blit(base, blend="add"); last = base
        fin = P("baseVertexShader", "bloomFinalShader")
        fin.set(texelSize=(last.texelSizeX, last.texelSizeY), uTexture=last, intensity=c["BLOOM_INTENSITY"])
        fin.blit(bloom)
    sw, sh = get_resolution(c["SUNRAYS_RESOLUTION"])
    mask = G.Texture(dye.w, dye.h, 4, True, half=True)
    sun, tmp = G.Texture(sw, sh, 1, True, half=True), G.Texture(sw, sh, 1, True, half=True)
    mp = P("baseVertexShader", "sunraysMaskShader"); mp.set(texelSize=(0.0, 0.0), uTexture=dye); mp.blit(mask)
    sp = P("baseVertexShader", "sunraysShader"); sp.set(texelSize=(0.0, 0.0), weight=c["SUNRAYS_WEIGHT"], uTexture=mask); sp.blit(sun)
    bp = P("blurVertexShader", "blurShader")
    bp.set(texelSize=(sun.texelSizeX, 0.0), uTexture=sun); bp.blit(tmp)
    bp.set(texelSize=(0.0, sun.texelSizeY), uTexture=tmp); bp.blit(sun)
    target = G.Texture(width, height, 4, True)
    col = P("baseVertexShader", "colorShader")
    col.set(texelSize=(1.0 / width, 1.0 / height), color=(back_color[0] / 255, back_color[1] / 255, back_color[2] / 255, 1))
    col.blit(target)
    dith = G.Texture(dither.shape[1], dither.shape[0], 3, True, repeat=True)
    dith.data[..., :3] = dither
    disp = P("baseVertexShader", "displayShaderSource", ("SHADING", "BLOOM", "SUNRAYS"))
    disp.set(texelSize=(1.0 / width, 1.0 / height), uTexture=dye, uBloom=bloom, uDithering=dith,
             ditherScale=(width / dith.w, height / dith.h), uSunrays=sun)          # S:1337-1346, S:1626-1631
    disp.blit(target, blend="premult")
    return dict(target=target.data.copy(), bloom=bloom.data.copy(), sunrays=sun.data[..., 0].copy(),
                mask_alpha=mask.data[..., 3].copy(), pyramid=[t.data.copy() for t in pyramid])


def postfx_half(name, Wd, Hd, w, h, seed, bloom_res=64, sun_res=48):
    from PIL import Image
    png = os.path.join(os.path.dirname(G.REFERENCE_JS), "LDR_LLL1_0.png")
    dither = np.asarray(Image.open(png).convert("RGB"), dtype=F) / F(255.0)
    rng = np.random.default_rng(seed)
    dye = (rng.random((Hd, Wd, 4), dtype=F) ** 4 * 3).astype(F); dye[..., 3] = 1     # as make_golden.py postfx()
    dye = dye.astype(np.float16).astype(F)
    r = executed_postfx_half(dye, w, h, dither, dict(BLOOM_RESOLUTION=bloom_res, SUNRAYS_RESOLUTION=sun_res), (10, 20, 30))
    o = dict(Wd=Wd, Hd=Hd, w=w, h=h, bloom_res=bloom_res, sun_res=sun_res, in_dye=dye, dither=dither.astype(np.float16),
             back=np.array([10, 20, 30], F), target=r["target"], bloom=r["bloom"].astype(F), sunrays=r["sunrays"],
             mask_alpha=r["mask_alpha"])
    for k, t in enumerate(r["pyramid"]):
        o[f"pyr{k}"] = t
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **o)


if __name__ == "__main__":
    postfx_half("postfx_half_64_to_128", 64, 64, 128, 128, 21)           # power-of-two target, dye and bloom FBO
    postfx_half("postfx_half_48x32_to_50x75", 48, 32, 50, 75, 22)        # ragged, portrait canvas
    print("half-storage post-FX golden vectors written to", OUT)
