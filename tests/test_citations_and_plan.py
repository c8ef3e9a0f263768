"""Housekeeping that needs no GPU: (1) every `S:n[-m]` citation in the product, oracle and docs points
inside the reference's script.js and, for the shader / function cites in include/fluid.h, at the
construct it names (against tests/golden/script_js_citations.json: the line count of script.js and
the lines on which each spot-check needle occurs, cut by tests/golden/make_golden.py citations);
(2) randomised invariants of the slab plan."""
import json
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_LINES = os.path.join(ROOT, "tests", "golden", "script_js_citations.json")
# (first line, last line, text that must occur on one of them) in script.js
SPOT_CHECKS = [
    (1231, 1294, "function step (dt)"), (1441, 1455, "function splat (x, y, dx, dy, color)"),
    (868, 890, "pressureShader"), (1259, 1266, "PRESSURE_ITERATIONS"),
    (746, 784, "advectionShader"), (786, 812, "divergenceShader"), (814, 833, "curlShader"),
    (835, 866, "vorticityShader"), (892, 913, "gradientSubtractShader"), (726, 744, "splatShader"),
    (508, 519, "clearShader"), (982, 1010, "function initFramebuffers"), (1612, 1624, "function getResolution"),
    (549, 612, "displayShaderSource"), (1296, 1317, "function render (target)"),
]
FILES = ["include/fluid.h", "DESIGN.md", "INTEGRATION.md", "oracle/fluid_oracle.c", "oracle/fluid_oracle.h",
         "oracle/glsl_exec.py", "webgl_fluid_simulation_b200/sim.py", "webgl_fluid_simulation_b200/js/fluid-sim.js",
         "webgl_fluid_simulation_b200/csrc/jacobi.cuh", "webgl_fluid_simulation_b200/csrc/passes.cuh",
         "webgl_fluid_simulation_b200/csrc/fluid.cu", "webgl_fluid_simulation_b200/csrc/stream_passes.cuh",
         "webgl_fluid_simulation_b200/csrc/half_passes.cuh", "webgl_fluid_simulation_b200/csrc/postfx.cuh",
         "webgl_fluid_simulation_b200/napi/fluid_napi.c", "README.md"]


def test_script_js_citations_are_in_range_and_on_target():
    ref = json.load(open(REF_LINES))
    n = ref["lines"]
    for f in FILES:
        for m in re.finditer(r"\bS:(\d+)(?:-(\d+))?", open(os.path.join(ROOT, f)).read()):
            a = int(m.group(1)); b = int(m.group(2) or a)
            assert 1 <= a <= b <= n, (f, m.group(0))
    # spot-check that the headline cites land on what they claim
    for lo, hi, needle in SPOT_CHECKS:
        assert any(lo <= k <= hi for k in ref["needle_lines"][needle]), (lo, hi, needle)


def test_slab_plan_invariants_randomised():
    from webgl_fluid_simulation_b200.slab import SlabPlan, jacobi_launches
    rng = np.random.default_rng(7)
    for _ in range(300):
        world = int(rng.integers(2, 9)); H = int(rng.integers(world * 16, 20000)); Hd = H * int(rng.choice([1, 2, 4]))
        iters = int(rng.integers(1, 90)); block = int(rng.integers(0, 14))
        try:
            plans = [SlabPlan(H, Hd, r, world, iterations=iters) for r in range(world)]
        except ValueError:
            assert H // world < 14
            continue
        assert plans[0].row0 == 0 and plans[-1].row1 == H and plans[-1].drow1 == Hd
        assert all(a.row1 == b.row0 and a.drow1 == b.drow0 for a, b in zip(plans, plans[1:]))       # a partition
        assert len({(p.G, p.Gd) for p in plans}) == 1                                                # same halo on every rank
        G = plans[0].G
        assert G <= min(p.row1 - p.row0 for p in plans)                                              # fits the shortest slab
        ks = jacobi_launches(iters, plans[0].block(block))
        assert sum(ks) == iters and max(ks) - min(ks) <= 1 and max(ks) <= 12
        for p in plans:
            ext = p.launch_extents(iters, block)
            assert [k for k, _ in ext] == ks and ext[-1][1] == 1                                     # gradient row
            if p.deep(iters):
                assert ext[0][1] + ext[0][0] == iters + 1 <= G                                       # first launch reads exactly the halo
                assert all(e0 - e1 == k1 for (_, e0), (k1, e1) in zip(ext, ext[1:]))                 # shrinks by the next depth
            else:
                assert max(k for k, _ in ext) + 1 <= G                                               # per-launch halo fits
