"""CPU reference of the post-FX chain in half-float storage (FLUID_FLAG_HALF_STORAGE).

The reference creates the bloom FBO, the bloom pyramid and both sunrays FBOs with
ext.halfFloatTexType (S:1012-1043) and draws the sunrays mask into the RGBA16F dye.write (S:1300),
so every post-FX blit rounds its output to fp16.  This is oracle.render_postfx with
oracle.round_half applied after every blit: prefilter, each down-sample, each additive up-sample
(fp32 add against the fp16 destination, then round), final, mask, march and both blur passes.
The final target stays fp32.  Built over the oracle's per-blit C functions; the fp32 chain of
oracle.render_postfx is left as it is.
"""
import ctypes as C

import numpy as np

from oracle import oracle as O


def _bind():
    L = O.lib(); i, f, p = C.c_int, C.c_float, O._f
    L.oracle_bloom_prefilter.argtypes = [p, i, i, p, i, i, f, f, f, f]
    L.oracle_box4.argtypes = [p, i, i, p, i, i, f, i]
    L.oracle_sunrays_mask.argtypes = [p, p, i, i]
    L.oracle_sunrays.argtypes = [p, i, i, p, i, i, f]
    L.oracle_blur3.argtypes = [p, p, i, i, f, f]
    L.oracle_display_full.argtypes = [p, i, i, p, i, i, p, i, i, p, i, i, p, i, i, p, i, f]
    for fn in (L.oracle_bloom_prefilter, L.oracle_box4, L.oracle_sunrays_mask, L.oracle_sunrays, L.oracle_blur3,
               L.oracle_display_full):
        fn.restype = None
    return L


def _round(a):
    """fp16 RN-even in place (oracle_round_half), so the caller's array stays the FBO."""
    O.lib().oracle_round_half(O._p(a), a.size)
    return a


def render_postfx_half(dye, w, h, dither, cfg=None, back_rgb=(0.0, 0.0, 0.0), background=0, aspect=None):
    """oracle.render_postfx with fp16 bloom / pyramid / mask / sunrays FBOs.  `dye` is the fp16 dye
    texture widened to fp32 (every value fp16-representable).  Returns the same keys."""
    L = _bind(); P = O._p
    c = dict(BLOOM_ITERATIONS=8, BLOOM_RESOLUTION=256, BLOOM_INTENSITY=0.8, BLOOM_THRESHOLD=0.6,
             BLOOM_SOFT_KNEE=0.7, SUNRAYS_RESOLUTION=196, SUNRAYS_WEIGHT=1.0)
    c.update(cfg or {})
    dye = O._c(dye); Hd, Wd, _ = dye.shape
    assert np.array_equal(dye, O.round_half(dye)), "the dye of a half-storage handle holds fp16 values"
    dither = O._c(dither)

    def get_resolution(res):                                  # S:1612-1624
        ar = w / h
        if ar < 1: ar = 1.0 / ar
        mn, mx = int(np.floor(res + 0.5)), int(np.floor(res * ar + 0.5))
        return (mx, mn) if w > h else (mn, mx)

    bw, bh = get_resolution(c["BLOOM_RESOLUTION"])
    bloom = np.zeros((bh, bw, 4), np.float32); bloom[..., 3] = 1.0        # createFBO clears to (0,0,0,1)
    sizes = []
    for k in range(c["BLOOM_ITERATIONS"]):
        pw, ph = bw >> (k + 1), bh >> (k + 1)
        if pw < 2 or ph < 2: break
        sizes.append((pw, ph))
    pyr = []
    if len(sizes) >= 2:
        knee = c["BLOOM_THRESHOLD"] * c["BLOOM_SOFT_KNEE"] + 0.0001
        L.oracle_bloom_prefilter(P(dye), Wd, Hd, P(bloom), bw, bh, c["BLOOM_THRESHOLD"] - knee, knee * 2,
                                 0.25 / knee, c["BLOOM_THRESHOLD"])
        _round(bloom)
        last, lw, lh = bloom, bw, bh
        for pw, ph in sizes:
            t = np.empty((ph, pw, 4), np.float32)
            L.oracle_box4(P(last), lw, lh, P(t), pw, ph, 1.0, 0)
            pyr.append(_round(t)); last, lw, lh = t, pw, ph
        for k in range(len(pyr) - 2, -1, -1):
            pw, ph = sizes[k]
            L.oracle_box4(P(last), lw, lh, P(pyr[k]), pw, ph, 1.0, 1)
            _round(pyr[k]); last, lw, lh = pyr[k], pw, ph
        L.oracle_box4(P(last), lw, lh, P(bloom), bw, bh, c["BLOOM_INTENSITY"], 0)
        _round(bloom)
    sw, sh = get_resolution(c["SUNRAYS_RESOLUTION"])
    mask = np.empty_like(dye)
    L.oracle_sunrays_mask(P(dye), P(mask), Wd, Hd)
    _round(mask)
    sun = np.empty((sh, sw), np.float32); tmp = np.empty_like(sun)
    L.oracle_sunrays(P(mask), Wd, Hd, P(sun), sw, sh, c["SUNRAYS_WEIGHT"])
    _round(sun)
    L.oracle_blur3(P(sun), P(tmp), sw, sh, 1.0 / sw, 0.0)
    _round(tmp)
    L.oracle_blur3(P(tmp), P(sun), sw, sh, 0.0, 1.0 / sh)
    _round(sun)
    out = np.empty((h, w, 4), np.float32)
    back = np.asarray(back_rgb, np.float32)
    L.oracle_display_full(P(dye), Wd, Hd, P(bloom), bw, bh, P(sun), sw, sh, P(dither), dither.shape[1],
                          dither.shape[0], P(out), w, h, P(back), int(background), float(w / h if aspect is None else aspect))
    return dict(target=out, bloom=bloom, sunrays=sun, mask_alpha=mask[..., 3].copy(), pyramid=pyr, mask=mask)
