#!/usr/bin/env python
"""bench.py — Jacobi pressure-solve throughput (BASELINE.json metric) on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the metric's hot path over one batch of synthetic input: the pressure
solve of step() — clear (p <- PRESSURE*p, S:1253-1257) + PRESSURE_ITERATIONS Jacobi sweeps
(S:1259-1266) — on BASELINE.json configs[2]: 4096x4096 fp32, 50 iterations, fields resident in HBM.
`value`    = W*H*iters*steps / device time (CUDA events on the library's own stream).
`parity`   = checked BEFORE timing, on the timed inputs, after three successive solves: temporally
             blocked == one-sweep-per-launch bit for bit, and at N>1 the CRC32 of every rank's owned
             rows == the same rows of a single-GPU run of the whole grid (the oracle comparison itself
             lives in tests/).
`e2e`      = the same solve through the C-ABI call with HOST buffers (fluid_pressure_solve_host:
             H2D divergence + pressure from pinned memory, solve, D2H pressure, all inside the call).
`e2e_step` = the drop-in frame: splat(...) -> step(dt) -> read dye into pinned host memory.
`roofline` is for the dominant kernel (jacobi_tb_kernel) on ALGORITHMIC bytes (12 B / update, SURVEY
§8d); temporal blocking moves far fewer DRAM bytes, so frac > 1 is expected and explained by
`jacobi_launches_per_step`, `compulsory_frac` and `traffic`; `roofline_naive` is the one-sweep-
per-launch kernel measured the same way (<= 1 by construction); `full_step.*.kernels` carries the
per-pass figures of a whole step().
`--impl reference`: the reference cannot run here (browser + WebGL, SURVEY §0.4), so the reference
arm is the CPU restatement of script.js (oracle/, kind "port") on the host cores this process may
use (affinity mask capped by the cgroup quota), buffers first-touched by the threads that sweep them.
`--dump-outputs DIR`: after the timed steps, the pressure field the last timed step left is written to
DIR/pressure.npy (float32; at N>1 DIR/pressure_rank<r>.npy, each rank its own rows), so that two builds
can be compared output for output on the same seeded inputs.  A field larger than the 32 MiB budget
(shared by the ranks) is cut to a fixed, seeded sample of its rows, whose indices go to
DIR/<name>_rows.npy (float64).
"""
from __future__ import annotations

import os


def _usable_cores() -> int:
    """Cores this process can really use: affinity mask capped by the cgroup CPU quota.  Taken
    FIRST: once an OpenMP runtime loads with OMP_PROC_BIND set it binds this thread to one core."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per) + 0.5)))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, int(q / per + 0.5)))
        except Exception:
            pass
    return n


USABLE_CORES = _usable_cores()
# the CPU legs use OpenMP: pin the team before ANY OpenMP runtime initialises (torch bundles one)
os.environ.setdefault("OMP_PROC_BIND", "close")
os.environ.setdefault("OMP_PLACES", "cores")

import argparse
import json
import sys
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def _baseline_metric():
    """BASELINE.json's own metric string (both arms print it verbatim)."""
    try:
        return json.load(open(os.path.join(ROOT, "BASELINE.json")))["metric"]
    except Exception:
        return "Jacobi cell-updates/sec at 4096²; achieved HBM GB/s vs B200 peak"


METRIC = _baseline_metric()     # `value` is the cell-updates/sec half; the GB/s half is `roofline.achieved`
UNIT = "cell-updates/s"
W = H = 4096
ITERS = 50
ALGO_BYTES_PER_UPDATE = 12  # read p 4 + read div 4 + write p 4 (SURVEY §8d)
DT = 0.016666
# algorithmic bytes per OUTPUT cell of the other passes (SURVEY §8d), fp32
PASS_BYTES = {"curl_vort_div": 24, "gradient": 20, "advect_velocity": 16, "advect_dye": 32}


def peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Polls NVML for SM clock + throttle reasons while the timed region runs."""

    def __init__(self, index, enabled=True, period=0.002):
        self.samples, self.reasons, self._stop = [], set(), threading.Event()
        self.period = period
        self.max_mhz = None
        try:
            if not enabled:
                raise RuntimeError("not the reporting rank")
            import pynvml as nv
            nv.nvmlInit()
            self.nv, self.h = nv, nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        names = {}
        for n in dir(nv):
            if n.startswith("nvmlClocksEventReason") or n.startswith("nvmlClocksThrottleReason"):
                v = getattr(nv, n)
                if isinstance(v, int) and v and (v & (v - 1)) == 0:
                    names.setdefault(v, n.replace("nvmlClocksEventReason", "").replace("nvmlClocksThrottleReason", ""))
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit and nm not in ("None", "GpuIdle", "ApplicationsClocksSetting"):
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(self.period)

    def __enter__(self):
        if self.nv:
            self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self.nv:
            self.t.join(timeout=1)

    def reset(self):
        self.samples = []; self.reasons = set()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unsampled"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def synth_inputs(seed=42, rows=None):
    """SURVEY §8d isolated-Jacobi inputs: div ~ U(-1,1) seed 42; p ~ N(0,1) so the decay pass has work."""
    rows = H if rows is None else rows
    rng = np.random.default_rng(seed)
    d = rng.uniform(-1, 1, (rows, W)).astype(np.float32)
    p = rng.standard_normal((rows, W)).astype(np.float32)
    return p, d


def crc(a: np.ndarray) -> int:
    return zlib.crc32(np.ascontiguousarray(a).view(np.uint8).reshape(-1).data)


DUMP_BYTES = 32 << 20     # --dump-outputs budget over all ranks


def dump_field(out_dir, name, a, budget):
    """a -> out_dir/name.npy as float32; above `budget` bytes only a fixed, seeded sample of its rows
    (sorted), with their indices in out_dir/name_rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    if a.nbytes > budget:
        k = max(1, budget // a[0].nbytes)
        rows = np.sort(np.random.default_rng(0).choice(a.shape[0], k, replace=False))
        np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
        a = a[rows]
    np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, np.float32))


# ---- CPU legs -------------------------------------------------------------------------------------

class CpuSolve:
    """The oracle's Jacobi loop on preallocated buffers that were FIRST-TOUCHED by the OpenMP team
    with the same static row schedule the sweeps use (so every thread sweeps pages of its own NUMA
    node), team sized to the cores this process can really use (oracle.usable_cores)."""

    def __init__(self):
        import ctypes as C
        from oracle import oracle as O
        self.O, self.L = O, O.lib()
        self.cores = O.use_all_cores(USABLE_CORES)       # torchrun exports OMP_NUM_THREADS=1
        p, d = synth_inputs()
        self.p, self.d, self.tmp = np.empty_like(p), np.empty_like(d), np.empty_like(p)
        fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
        self.fp = fp
        self.L.oracle_copy_rows(fp(self.p), fp(p), W, H)         # parallel first touch
        self.L.oracle_copy_rows(fp(self.d), fp(d), W, H)
        self.L.oracle_copy_rows(fp(self.tmp), fp(p), W, H)

    def sweeps(self, n):
        self.L.oracle_jacobi_iters(self.fp(self.p), self.fp(self.tmp), self.fp(self.d), W, H, n)


def cpu_port_rate(samples=5, sweeps=10):
    """CPU restatement of the pressure loop on a bounded sample, best-of-`samples`."""
    c = CpuSolve()
    c.sweeps(2)                                          # warm-up, page in
    ts = []
    for _ in range(samples):
        t0 = time.perf_counter(); c.sweeps(sweeps); ts.append(time.perf_counter() - t0)
    rates = [W * H * sweeps / t for t in ts]
    return {"value": max(rates), "median": float(np.median(rates)), "min": min(rates), "unit": UNIT,
            "cores": c.cores, "kind": "port",
            "sample": f"best of {samples} timings of {sweeps} Jacobi sweeps of {W}x{H} fp32 (= {sweeps / ITERS:.1f} x the "
                      f"{ITERS}-sweep solve), {sum(ts):.1f} s of CPU time; OpenMP team = usable cores "
                      f"(affinity mask capped by the cgroup quota), first-touch by the sweeping threads"}


def run_reference(args, rank, world):
    """Reference arm: the reference's own WebGL path cannot run here (SURVEY §0.4), so this is the CPU
    restatement of its pressure loop (oracle/, C + OpenMP) on the same inputs.  Each step is a
    bounded sample: SWEEPS Jacobi sweeps of the 50-sweep solve, on preallocated, first-touched
    buffers (no per-step allocation or copies in the timed region)."""
    if rank != 0:
        return
    c = CpuSolve()
    sweeps = 10                                          # bounded sample per step (even: result lands back in p)
    for _ in range(max(args.warmup, 3)):
        c.sweeps(2)
    per = []
    t_all = time.perf_counter()
    for _ in range(args.steps):
        t0 = time.perf_counter(); c.sweeps(sweeps); per.append(time.perf_counter() - t0)
    dt = time.perf_counter() - t_all
    if args.dump_outputs:
        dump_field(args.dump_outputs, "pressure", c.p, DUMP_BYTES)
    val = W * H * sweeps * args.steps / dt
    rates = [W * H * sweeps / t for t in per]
    sample = f"each step = {sweeps} Jacobi sweeps of {W}x{H} fp32 out of the {ITERS}-sweep solve"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": workload_config(world, None, False),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": c.cores, "kind": "port", "sample": sample,
                         "best_step": max(rates), "median_step": float(np.median(rates)), "worst_step": min(rates),
                         "note": "CPU restatement of script.js (oracle/, OpenMP); the WebGL reference cannot run "
                                 "in this image (no browser / GL / node)"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def workload_config(world, transport, strong):
    """Identical keys in both arms (the driver compares the dicts)."""
    return {"workload": f"pressure solve {W}x{W} fp32, {ITERS} Jacobi iterations" + (" (BASELINE configs[2])" if (W, ITERS) == (4096, 50) else ""),
            "l2": f"working set {12 * W * H / 2**20:.0f} MiB per GPU (p x2 + div) vs 126 MB L2; no explicit flush between steps",
            "parallelism": "single GPU" if world == 1 else
            (f"{world} row slabs; weak: every GPU owns {W}x{H} of a {W}x{H * world} grid" if not strong else
             f"{world} row slabs of ONE {W}x{W} grid") + "; one deep halo exchange per solve"}


HOST_MS = {}


def time_steps(sim, fn, steps, tag=None, align=False):
    # align (N>1): one untimed solve between the barrier and the start event.  A solve on slabs is a collective
    # between neighbours, so it lines the ranks up ON THE DEVICE: host-side skew after the barrier (a process
    # that gets the CPU a few milliseconds late) would otherwise sit inside its neighbours' device timers, as
    # they spin in the halo exchange waiting for it (seen at N=8: a constant 40-75 ms per run, whatever --steps).
    if align:
        fn()
    sim.mark(0)
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    host = time.perf_counter() - t0          # enqueue time only: if it approaches the device time the run is host-bound
    sim.mark(1)
    ms = sim.elapsed_ms()
    if tag:
        HOST_MS[tag] = 1e3 * host / steps
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--jacobi-block", type=int, default=0)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--quick", action="store_true", help="timed region only (tuning runs): no parity / e2e / naive / full-step / cpu legs")
    ap.add_argument("--grid", type=int, default=4096, help="square grid size of the workload (BASELINE configs: 4096 / 8192 / 16384)")
    ap.add_argument("--iters", type=int, default=50, help="Jacobi iterations per solve (BASELINE configs: 50 / 40 / 80)")
    ap.add_argument("--strong", action="store_true", help="N>1: the headline `value` is measured on ONE grid x grid domain split into N row slabs (default: weak, one grid x grid slab per GPU, plus a `strong` block)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the pressure field of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    global W, H, ITERS
    W = H = args.grid
    ITERS = args.iters

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch
    import webgl_fluid_simulation_b200 as pkg
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the library has no CPU path")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        from webgl_fluid_simulation_b200.distributed import create_slab_simulation

    cfg = {"SIM_RESOLUTION": W, "DYE_RESOLUTION": 64, "PRESSURE_ITERATIONS": ITERS}
    strong_main = world > 1 and args.strong
    rows = args.grid // world if strong_main else args.grid     # rows this rank owns
    H = rows
    p0, d0 = synth_inputs(42 + rank, rows)               # every rank its own slab of the global input

    def make_sim(flags=0, jb=args.jacobi_block, rows_per_rank=rows):
        if world == 1:
            return pkg.FluidSimulation(cfg, 1024, 1024, device=local, flags=flags, jacobi_block=jb)
        return create_slab_simulation(cfg, 1024, 1024, device=local, flags=flags, jacobi_block=jb,
                                      # the (unused) dye grid is tiny; its rows per rank bound the ghost zone, which must
                                      # hold ITERS + 2 rows for the one-exchange-per-solve schedule
                                      sizes=(W, rows_per_rank * world, 64, max(64, ITERS + 2) * world))

    sim = make_sim()
    transport = getattr(sim, "halo_transport", None)

    def load(s, p=p0, d=d0):
        s.writeField("pressure", p); s.writeField("divergence", d)

    def barrier():
        sim.sync(); torch.cuda.synchronize()
        if dist: dist.barrier()
        torch.cuda.synchronize()

    # ---- parity, BEFORE timing, on the timed inputs ------------------------------------------------
    parity = None
    if not args.quick:
        parity = {}
        # THREE successive solves (each one: clear pass + the Jacobi loop on the previous result), so that the
        # steady state of the timed loop is what is compared — on slabs, solves 2 and 3 start from ghost rows
        # that are already in place (divergence not re-sent; pressure rows stored by the neighbour's last launch)
        def solve3(s_):
            for _ in range(3):
                s_.pass_("pressure_solve")
        load(sim); solve3(sim); mine = sim.readField("pressure")
        nsim = make_sim(flags=pkg.FLAG_NAIVE_JACOBI, jb=1)
        load(nsim); solve3(nsim); naive = nsim.readField("pressure"); nsim.close()
        same = bool(np.array_equal(mine.view(np.uint32), naive.view(np.uint32)))
        del naive
        if dist:
            t = torch.tensor([1 if same else 0], device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MIN); same = bool(t.item())
        parity["blocked_eq_naive_bitwise"] = same
        if world > 1:
            crcs = [None] * world
            dist.all_gather_object(crcs, crc(mine))
            ok = None
            if rank == 0:
                # the whole W x (rows*world) grid on ONE GPU (rank 0's), same library, single-GPU path
                gp = np.concatenate([synth_inputs(42 + r, rows)[0] for r in range(world)], axis=0)
                gd = np.concatenate([synth_inputs(42 + r, rows)[1] for r in range(world)], axis=0)
                one = pkg.FluidSimulation(cfg, 1024, 1024, device=local, jacobi_block=args.jacobi_block,
                                          sizes=(W, rows * world, 64, 64 * world))
                one.writeField("pressure", gp); one.writeField("divergence", gd)
                solve3(one); full = one.readField("pressure"); one.close()
                ok = all(crc(full[r * rows:(r + 1) * rows]) == crcs[r] for r in range(world))
                del gp, gd, full
            box = [ok]
            dist.broadcast_object_list(box, src=0)
            parity["slabs_eq_single_gpu_bitwise"] = bool(box[0])
            parity["slabs_check"] = (f"CRC32 of every rank's owned rows ({W}x{rows}) after 3 successive solves vs the same rows "
                                     f"of a single-GPU run of the {W}x{rows * world} grid on rank 0's GPU")
        parity["solves"] = 3
        del mine
        load(sim)

    load(sim)
    solve = lambda: sim.pass_("pressure_solve")
    # NVML is initialised (and its polling thread started) BEFORE the warm-up and the barrier: nvmlInit with 8
    # processes on one box takes milliseconds, which must not sit between the barrier and the timed region.
    # Only rank 0 reports clocks, so only rank 0 polls.
    with ClockSampler(local, enabled=(rank == 0), period=0.002 if world == 1 else 0.005) as clk:
        for _ in range(args.warmup):
            solve()
        barrier()
        clk.reset()                       # keep only the samples taken during the timed region
        ms = time_steps(sim, solve, args.steps, tag="solve", align=world > 1)
        sim.sync()
        # read before the extra solves below overwrite it; written once the clock sampler has stopped
        dumped = sim.readField("pressure") if args.dump_outputs else None
        # keep the device loaded until NVML has a few samples even if the timed region is short
        # (single GPU only: on slabs every solve is a collective, so all ranks must issue the
        # same number of them; there a fixed number of extra solves keeps the sampler fed)
        if world == 1:
            t_end = time.time() + 0.25
            while len(clk.samples) < 5 and time.time() < t_end:
                solve(); sim.sync()
        else:
            for _ in range(20):
                solve()
            sim.sync()
    if dumped is not None:
        dump_field(args.dump_outputs, "pressure" if world == 1 else f"pressure_rank{rank}", dumped, DUMP_BYTES // world)
        del dumped
    barrier()
    # exact launch counts of the timed region: kernels per solve x steps, Jacobi kernels separately
    l1, j1, h1 = sim.launch_count(), sim.stat("jacobi_launches"), sim.stat("halo_launches")
    solve(); sim.sync()
    per_step_launches = sim.launch_count() - l1
    jacobi_per_step = sim.stat("jacobi_launches") - j1
    halo_per_step = sim.stat("halo_launches") - h1
    gpu_launches = per_step_launches * args.steps
    if dist:
        t = torch.tensor([ms], device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
    value = W * H * ITERS * args.steps * world / (ms * 1e-3)     # all ranks' cells / max-over-ranks time

    peak, peak_src = peak_hbm()
    achieved = ALGO_BYTES_PER_UPDATE * W * H * ITERS * args.steps / (ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "jacobi_traffic.json")
    if os.path.exists(tp) and world == 1 and (W, ITERS) == (4096, 50):
        try:
            tj = json.load(open(tp))
            traffic = tj.get("dram_bytes_per_launch")
            traffic_src = tj.get("source", "profiles/jacobi_traffic.json") + " (one ncu --set full capture of this kernel at this size; NOT re-measured in this run)"
        except Exception:
            traffic = None
    sm_mhz = clk.summary().get("sm_mhz") or 1965.0
    roofline = {
        "kernel": "jacobi_tb_kernel", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
        "algorithmic_bytes_per_update": ALGO_BYTES_PER_UPDATE,
        "jacobi_launches_per_step": jacobi_per_step, "halo_kernels_per_step": halo_per_step,
        "avg_launch_ms": ms / (args.steps * max(jacobi_per_step, 1)),
        "avg_launch_note": "timed region / Jacobi launches" + ("" if world == 1 else "; at N>1 the region also holds one halo exchange per solve"),
        "algorithmic_bytes_per_launch": ALGO_BYTES_PER_UPDATE * W * H * ITERS / max(jacobi_per_step, 1),
        "updates_per_launch": W * H * ITERS / max(jacobi_per_step, 1),
        "compulsory_frac": (ALGO_BYTES_PER_UPDATE * W * H * jacobi_per_step * args.steps / (ms * 1e-3) / 1e9) / peak,
        "note": "per GPU.  Temporal blocking runs several sweeps per launch out of registers, so the "
                "12 B/update algorithmic figure exceeds what DRAM actually moves; frac > 1 is "
                "expected; compulsory_frac counts 12 B/cell once per Jacobi launch",
        # what actually bounds the blocked kernel: fp32 lane-operations on the 128 lanes/SM (the packed
        # f32x2 forms save issue slots, not lane-cycles); 4 ops/update with the contracted tail
        "fp32_pipe": {"ops_per_update": 4,
                      "achieved_tops": 4 * W * H * ITERS * args.steps / (ms * 1e-3) / 1e12,
                      "peak_tops": 148 * 128 * (sm_mhz * 1e6) / 1e12,
                      "frac": (4 * W * H * ITERS * args.steps / (ms * 1e-3)) / (148 * 128 * (sm_mhz * 1e6)),
                      "note": "useful updates only; overlapped tiling recomputes part of them (x halo columns, y warm-up rows per chunk)"},
    }

    cfgd = workload_config(world, transport, strong_main)
    if world > 1:
        cfgd["halo"] = f"{ITERS + 1} rows of p + {ITERS} of div per neighbour per solve, transport {transport}"
        cfgd["rank_alignment"] = ("one untimed solve (a neighbour-collective) between the barrier and the start event lines the "
                                  "ranks up on the device; the K timed solves follow it, max over ranks")
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "strong" if strong_main else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfgd,
        "clocks": clk.summary(), "gpu_launches": gpu_launches, "roofline": roofline,
        "host_enqueue_ms_per_step": HOST_MS.get("solve"),
    }
    if parity is not None:
        out["parity"] = parity

    if args.quick:
        if rank == 0:
            print(json.dumps(out))
        sim.close()
        if dist:
            dist.barrier(); dist.destroy_process_group()
        return
    # ---- e2e: host buffers through the C ABI; every rank moves its own slab -----------------------
    ph = torch.empty((H, W), dtype=torch.float32).pin_memory()
    dh = torch.empty((H, W), dtype=torch.float32).pin_memory()
    ph.numpy()[...] = p0; dh.numpy()[...] = d0
    pn, dn = ph.numpy(), dh.numpy()
    e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        sim.pressure_solve_host(dn, pn, ITERS)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e_steps):
        sim.pressure_solve_host(dn, pn, ITERS)
    e_dt = time.perf_counter() - t0
    if dist:
        t = torch.tensor([e_dt], device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX); e_dt = float(t.item())
    out["e2e"] = {"value": W * H * ITERS * e_steps * world / e_dt, "unit": UNIT,
                  "h2d_bytes_per_step": 2 * W * H * 4 * world, "d2h_bytes_per_step": W * H * 4 * world,
                  "ms_per_step": 1e3 * e_dt / e_steps, "steps": e_steps,
                  "api": "fluid_pressure_solve_host (pinned host buffers; H2D div+p, solve, D2H p, all inside the call; one GPU: row bands solved and downloaded behind the upload; per rank: its slab)"}
    del ph, dh

    # ---- strong scaling of the headline grid (north_star: "1/2/4/8 B200 on a 4096^2 grid") ----------
    if world > 1 and not strong_main:
        srows = args.grid // world
        ssim = make_sim(rows_per_rank=srows)
        sp, sd = synth_inputs(42, srows)
        ssim.writeField("pressure", sp); ssim.writeField("divergence", sd)
        ssolve = lambda: ssim.pass_("pressure_solve")
        for _ in range(args.warmup): ssolve()
        ssim.sync(); dist.barrier()
        sms = time_steps(ssim, ssolve, args.steps, align=True); ssim.sync()
        t = torch.tensor([sms], device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX); sms = float(t.item())
        out["strong"] = {"value": W * args.grid * ITERS * args.steps / (sms * 1e-3), "unit": UNIT, "ms_per_step": sms / args.steps,
                         "grid": f"ONE {W}x{args.grid} grid split into {world} row slabs of {srows} rows", "steps": args.steps,
                         "halo_bytes_per_exchange_per_neighbour": (2 * ITERS + 1) * W * 4}
        ssim.close()

    if rank == 0 and world == 1:
        # ---- naive (one sweep per launch) kernel, same inputs, same timing method ----------------
        nsim = pkg.FluidSimulation(cfg, 1024, 1024, device=local, flags=pkg.FLAG_NAIVE_JACOBI, jacobi_block=1)
        nsim.writeField("pressure", p0); nsim.writeField("divergence", d0)
        nsolve = lambda: nsim.pass_("pressure_solve")
        for _ in range(3): nsolve()
        nsim.sync()
        nsteps = max(3, min(args.steps, 20))
        nms = time_steps(nsim, nsolve, nsteps); nsim.sync()
        nach = ALGO_BYTES_PER_UPDATE * W * H * ITERS * nsteps / (nms * 1e-3) / 1e9
        out["roofline_naive"] = {"kernel": "jacobi_sweep_kernel", "bound": "hbm", "achieved": nach, "peak": peak,
                                 "unit": "GB/s", "frac": nach / peak, "ms_per_step": nms / nsteps,
                                 "updates_per_s": W * H * ITERS * nsteps / (nms * 1e-3)}
        nsim.close()
        # ---- half-float storage (the reference's own texture format, S:138-147): 6 B per update ---------
        hsim = pkg.FluidSimulation(cfg, 1024, 1024, device=local, flags=pkg.FLAG_HALF_STORAGE)
        hsim.writeField("pressure", p0); hsim.writeField("divergence", d0)
        hsolve = lambda: hsim.pass_("pressure_solve")
        for _ in range(3): hsolve()
        hsim.sync()
        hsteps = max(3, min(args.steps, 20))
        hms = time_steps(hsim, hsolve, hsteps); hsim.sync()
        hach = 6 * W * H * ITERS * hsteps / (hms * 1e-3) / 1e9
        out["roofline_half_storage"] = {"kernel": "hs::jacobi8_kernel (one sweep per launch, fp16 fields, fp32 arithmetic, RN-even on write)",
                                        "bound": "hbm", "algorithmic_bytes_per_update": 6, "achieved": hach, "peak": peak, "unit": "GB/s",
                                        "frac": hach / peak, "ms_per_step": hms / hsteps, "updates_per_s": W * H * ITERS * hsteps / (hms * 1e-3)}
        hsim.close()

        # ---- whole step() on configs[1] and configs[2], with per-pass rooflines ------------------------
        ctx = {}
        for name, c in (("1024x1024 sim / 2048x2048 dye, 30 iters", {"SIM_RESOLUTION": 1024, "DYE_RESOLUTION": 2048, "PRESSURE_ITERATIONS": 30}),
                        ("4096x4096 sim / 4096x4096 dye, 50 iters", {"SIM_RESOLUTION": 4096, "DYE_RESOLUTION": 4096, "PRESSURE_ITERATIONS": 50})):
            s2 = pkg.FluidSimulation(c, 1024, 1024, device=local, flags=pkg.FLAG_NO_GRAPH, random=np.random.RandomState(1234).random_sample)
            s2.multipleSplats(16)
            for _ in range(3): s2.step(DT)
            n2 = 10
            acc = {}
            m2 = 0.0
            for _ in range(n2):                           # per-pass CUDA events of every step, averaged
                m2 += time_steps(s2, lambda: s2.step(DT), 1); s2.sync()
                for k, v in s2.timing().items():
                    acc[k] = acc.get(k, 0.0) + v
            tm = {k: v / n2 for k, v in acc.items()}
            sw, dw = c["SIM_RESOLUTION"], c["DYE_RESOLUTION"]
            kern = {}
            for pname, nbytes in PASS_BYTES.items():
                cells = dw * dw if pname == "advect_dye" else sw * sw
                extra = 8 * sw * sw if pname == "advect_dye" else 0          # + the velocity field read once
                t_ms = tm[pname + "_ms"]
                gbs = (nbytes * cells + extra) / (t_ms * 1e-3) / 1e9
                kern[pname] = {"ms": round(t_ms, 4), "algorithmic_bytes_per_cell": nbytes, "achieved_gbs": round(gbs, 1), "frac": round(gbs / peak, 3)}
            ctx[name] = {"ms_per_step": m2 / n2, "passes_ms": {k: round(v, 4) for k, v in tm.items() if k.endswith("_ms")},
                         "kernels": kern, "launches_per_step": int(tm["total_launches"])}
            s2.close()
        out["full_step"] = ctx
        # ---- the reference's own default config (launch-bound regime): graph replay vs pass by pass ----
        dflt = {}
        for tag, fl in (("cuda_graph", 0), ("pass_by_pass", pkg.FLAG_NO_GRAPH)):
            s3 = pkg.FluidSimulation({}, 1024, 1024, device=local, flags=fl, random=np.random.RandomState(7).random_sample)
            s3.multipleSplats(8)
            for _ in range(5): s3.step(DT)
            n3 = 200
            m3 = time_steps(s3, lambda: s3.step(DT), n3); s3.sync()
            dflt[tag] = {"ms_per_step": m3 / n3}
            if tag == "cuda_graph":
                # the reference's frame loop: a different dt on every frame (calcDeltaTime S:1188-1194)
                rng = np.random.default_rng(3)
                dts = [float(x) for x in rng.uniform(0.004, 0.016666, n3)]
                it = iter(dts)
                c0 = s3.stat("graph_captures")
                m4 = time_steps(s3, lambda: s3.step(next(it)), n3); s3.sync()
                dflt["cuda_graph_jittered_dt"] = {"ms_per_step": m4 / n3, "graph_captures_during": s3.stat("graph_captures") - c0}
            s3.close()
        out["default_config_step"] = {"config": "128x128 sim / 1024x1024 dye, 20 iters (script.js defaults, S:59-69)", **dflt,
                                      "reference_draw_calls_per_step": 27, "kernels_per_step": 6}

        # ---- e2e of the drop-in frame: splat -> step -> read dye (pinned host buffer) -----------------
        s4 = pkg.FluidSimulation({"SIM_RESOLUTION": 4096, "DYE_RESOLUTION": 4096, "PRESSURE_ITERATIONS": ITERS}, 1024, 1024,
                                 device=local, random=np.random.RandomState(99).random_sample)
        dye_host = torch.empty((4096, 4096, 4), dtype=torch.float32).pin_memory()
        dyn = dye_host.numpy()
        s4.multipleSplats(4)
        for _ in range(2):
            s4.splat(0.5, 0.5, 300.0, -200.0, (0.3, 0.1, 0.9)); s4.step(DT); s4.readField("dye", out=dyn)
        n4 = 5
        t0 = time.perf_counter()
        for k in range(n4):
            s4.splat(0.2 + 0.1 * k, 0.6, 300.0, -200.0, (0.3, 0.1, 0.9)); s4.step(DT); s4.readField("dye", out=dyn)
        f_dt = time.perf_counter() - t0
        out["e2e_step"] = {"value": 4096 * 4096 * ITERS * n4 / f_dt, "unit": UNIT, "ms_per_frame": 1e3 * f_dt / n4, "frames_per_s": n4 / f_dt,
                           "h2d_bytes_per_step": 7 * 4, "d2h_bytes_per_step": 4096 * 4096 * 16, "steps": n4,
                           "api": "splat(x,y,dx,dy,color) -> step(dt) -> readField('dye') into pinned host memory "
                                  "(4096x4096 sim and dye, 50 iterations): the call sequence of the reference's update() + render input"}
        s4.close()
        del dye_host

        if not args.no_cpu:
            out["cpu_baseline"] = cpu_port_rate()
    if rank == 0:
        print(json.dumps(out))
    sim.close()
    if dist:
        dist.barrier(); dist.destroy_process_group()


if __name__ == "__main__":
    main()
