#!/usr/bin/env python
"""bench.py -- Gauss-Newton Mpix-iters/s of the SMVS depth-refinement hot path.

Headline workload (BASELINE.json configs[1]): 1 reference view + 6 neighbours,
1920x1080, finest scale of `-o2` (scale 2: 478x268 patches of 4x4 px, 16
samples each, every pixel sampled), no shading. One STEP = one inner Newton
loop of DepthOptimizer::run_newton_iterations (lib/depth_optimizer.cc:204-304:
construct -> PCG -> node update / active set, repeated until < 5 % of the nodes
are active) of ONE view, started from its 2 % perturbed surface. A
pixel-iteration is one sample of one processed patch in one Newton step
(SURVEY.md section 8d).

  value  pixel-iterations / device time of the loop (CUDA events on the
         library's stream, inputs resident in HBM)
  e2e    the same loop through the C ABI from HOST buffers, every step:
         smvsb_set_views_u8 (H2D of the 7 byte images from pinned memory +
         StereoView::set_scale on the device) + smvsb_set_surface (H2D of nodes,
         validity, visibility) + smvsb_newton_loop + smvsb_get_nodes (D2H),
         wall clock around the calls with a device synchronize on both sides

Views. The work of a loop depends on the view (its active set shrinks at its
own pace), so every rank cycles through the same pool of POOL = 4 seeded views
(rank r starts at view r mod 4): per-GPU work is the same on every rank and at
every N ("weak" scaling in the strict sense), different GPUs work on different
views at any one time, and there is no data-path collective -- reference views
are independent units (app/smvsrecon.cc:658-733).

`configs` (same JSON line) carries the other BASELINE.json configurations, each
with its own roofline and (N = 1) cpu_baseline:
  shading       configs[2]: the same loop with -S (lighting fitted per view)
  sgm           configs[3]: SGM 1920x1080, 128 planes, 8 paths (N = 1 only)
  batch4        configs[4]: 4 views per GPU with -S, their Newton loops run in
                lock-step with ONE persistent PCG launch per step
                (smvsb_newton_loop_batch); value = all ranks' pixel-iterations
                / max-over-ranks time

--impl reference times the reference's own CPU implementation (oracle/_ref:
the reference's sources compiled verbatim against the MVE shim) the way the
reference parallelises: one view per host thread (its ThreadPool,
app/smvsrecon.cc:558,658-733). Each thread owns a REAL small view (480x270, 6
neighbours, its own node grid, scale 2) -- a bounded sample of the same
workload whose size does not depend on --steps; the thread count is the one
that gives the reference its best throughput on this host (calibrated before
the warm-up, or SMVSB_REF_THREADS).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from smvs_b200.workload import build_workload  # noqa: E402,F401  (tests import it from here)

WIDTH, HEIGHT, N_SUB, SCALE = 1920, 1080, 6, 2
POOL = 4                        # views a rank cycles through
BATCH = 4                       # views per GPU of configs[4]
SMALL_W, SMALL_H = 480, 270     # the CPU arms' bounded sample: one real small view
SMALL_POOL = 8
REGULARIZATION = 0.01           # app/smvsrecon.cc:712 with alpha = 1
METRIC = "Gauss-Newton Mpix-iters/sec"
DUMP_STATS = ("newton_steps", "cg_iterations", "pixel_iterations", "n_active")
DUMP_LIMIT = 64 << 20           # bytes of --dump-outputs
UNIT = "Mpix-iters/s"
CONFIG = {
    "workload": "1 ref view + 6 neighbours, 1920x1080, scale 2 (-o2), no shading: "
                "inner Newton loop of one view from its 2% perturbed surface",
    "views": f"pool of {POOL} seeded views, every rank cycles through all of them",
    "views_per_gpu_in_flight": 1,
    "l2": "inputs_exceed_l2 (packed images 415 MB, H 148 MB per view)",
}


# ---------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------

class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                 "-i", str(self.index), "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t_begin=None, t_end=None):
        """Samples that arrived inside [t_begin, t_end] (the timed region); the
        sampler is started before the warm-up because nvidia-smi needs a few
        hundred ms to produce its first line."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lines = [ln for (t, ln) in self.lines
                 if t_begin is None or (t_begin <= t <= t_end + 0.05)]
        if not lines:          # region shorter than the sampling jitter: nearest ones
            lines = [ln for (_, ln) in self.lines[-5:]]
        for ln in lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(smax)) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------
# workloads (built in forked worker processes, before CUDA is touched)
# ---------------------------------------------------------------------------

def _build_one(spec):
    w, h, n_sub, scale, shading, seed = spec
    return build_workload(w, h, n_sub, scale, shading=shading, seed_index=seed)


def build_pool(specs):
    """Workloads for the given (w, h, n_sub, scale, shading, seed) specs, built
    concurrently (numpy host code, ~10 s each at 2 MP)."""
    import multiprocessing as mp
    if len(specs) <= 1 or (os.cpu_count() or 1) < 2:
        return [_build_one(s) for s in specs]
    ctx = mp.get_context("fork")
    with ctx.Pool(min(len(specs), os.cpu_count() or 1)) as pool:
        return pool.map(_build_one, specs)


# ---------------------------------------------------------------------------
# CPU arms (oracle used as the thing timed ONLY here, as the task allows)
# ---------------------------------------------------------------------------

def _ref_scene_for(wl):
    """A reference DepthOptimizer state fed with exactly the workload's
    prepared arrays."""
    from oracle import ref as oref
    R = oref.RefScene(wl.scene, init_linear=wl.shading is not None)
    R.set_arrays(0, wl.main_grad, None)
    for k in range(wl.scene.n_sub):
        R.set_arrays(k + 1, wl.sub_grads[k], wl.sub_hess[k])
    if wl.shading is not None:
        R.set_shading(wl.shading, wl.shading_grad)
    R.surface_create(wl.scale, np.full((wl.scene.height, wl.scene.width), 5.0, np.float32))
    info = R.surface_info()
    assert (info["npx"], info["npy"], info["start_x"], info["start_y"]) == \
        (wl.npx, wl.npy, wl.start_x, wl.start_y)
    R.surface_set(wl.nodes, wl.node_valid, wl.patch_valid)
    R.set_visibility(wl.vis_off, wl.vis_ids)
    return R


class ReferenceWorkers:
    """`threads` reference optimizers, each on its own real small view (one
    of `pool`, round robin); run() lets every one do one Newton loop
    concurrently, one host thread each (the reference's ThreadPool model: one
    view per thread, app/smvsrecon.cc:558,658-733)."""

    def __init__(self, pool, threads, shading=False):
        from oracle import ref as oref
        if not oref.available():
            raise RuntimeError("oracle/_ref missing")
        self.threads = threads
        self.subs = [pool[i % len(pool)] for i in range(threads)]
        self.scenes = [_ref_scene_for(sub) for sub in self.subs]
        self.lights = [None] * threads
        if shading:
            self.lights = [R.fit_lighting() for R in self.scenes]
        wl = pool[0]
        self.desc = (f"one real {wl.scene.width}x{wl.scene.height} view with {wl.scene.n_sub} "
                     f"neighbours per host thread (own {wl.npx}x{wl.npy}-patch grid, scale "
                     f"{wl.scale}{', -S' if shading else ''}), one inner Newton loop each per step")

    def run(self, n_threads=None, repeats=1):
        n = n_threads or self.threads
        results = [0.0] * n

        def work(i):
            R, sub = self.scenes[i], self.subs[i]
            for _ in range(repeats):
                R.surface_set(sub.nodes, sub.node_valid, sub.patch_valid)
                st = R.newton_loop(self.lights[i], REGULARIZATION, 0.0)
                results[i] += st["pixel_iterations"]

        t0 = time.perf_counter()
        th = [threading.Thread(target=work, args=(i,)) for i in range(n)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        return float(sum(results)), time.perf_counter() - t0

    def run_serial(self):
        """Every view's loop once, one after the other on the calling thread."""
        pix = 0.0
        t0 = time.perf_counter()
        for R, sub, light in zip(self.scenes, self.subs, self.lights):
            R.surface_set(sub.nodes, sub.node_valid, sub.patch_valid)
            pix += R.newton_loop(light, REGULARIZATION, 0.0)["pixel_iterations"]
        return pix, time.perf_counter() - t0

    def close(self):
        for R in self.scenes:
            R.close()


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return 0
    ncpu = os.cpu_count() or 1
    pool = build_pool([(SMALL_W, SMALL_H, N_SUB, SCALE, False, s) for s in range(SMALL_POOL)])
    forced = int(os.environ.get("SMVSB_REF_THREADS", "0"))
    cands = [forced] if forced > 0 else sorted({t for t in (8, 16, 32, 64, 128, ncpu)
                                                if t <= ncpu} or {1})
    workers = ReferenceWorkers(pool, max(cands))
    # the reference's throughput stops growing with threads early (every vector
    # operation of its CG allocates, and the threads share one address space):
    # take the thread count that serves it best on this host
    calib = {}
    for t in cands:
        p, s = workers.run(t)
        calib[t] = p / s / 1e6
    threads = max(calib, key=calib.get)
    for _ in range(args.warmup):
        workers.run(threads)
    pix, secs = 0.0, 0.0
    for _ in range(args.steps):
        p, s = workers.run(threads)
        pix += p
        secs += s
    desc = workers.desc
    workers.close()
    value = pix / secs / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * secs / max(args.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": dict(CONFIG),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads,
                         "kind": "reference", "sample": desc,
                         "host_cpus": ncpu,
                         "threads_calibration_mpix_iters_s": {str(k): v for k, v in calib.items()}},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------
# product arm
# ---------------------------------------------------------------------------

def _system_blocks_full(wl):
    """4x4 blocks of the full system (every valid node active)."""
    nv = wl.node_valid.reshape(wl.npy + 1, wl.npx + 1).astype(bool)
    blocks = 0
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            a = nv[max(dy, 0):nv.shape[0] + min(dy, 0), max(dx, 0):nv.shape[1] + min(dx, 0)]
            b = nv[max(-dy, 0):nv.shape[0] + min(-dy, 0), max(-dx, 0):nv.shape[1] + min(-dx, 0)]
            blocks += int((a & b).sum())
    return blocks


# fp64 operations (DADD + DMUL + 2 DFMA, as executed) of gn_patch_kernel<16> per
# pixel-iteration at 6 visible neighbours, no shading term: from the ncu capture
# named below (smsp__sass_thread_inst_executed_op_{dadd,dmul,dfma}_pred_on.sum of
# one launch / its samples). This is the basis-space formulation's work -- the
# reference's 16-wide rank-1 formulation would be ~20 kFLOP (SURVEY.md section 8d).
# Captured launch (final kernel of round 2, divisions by d, d^2, d^4 through one
# reciprocal): 5.074e9 DFMA + 3.088e9 DMUL + 1.563e9 DADD thread instructions for
# 118 326 processed patches x 16 pixels. 48 % of the fp64 instructions are not
# fused (the bitwise-parity arithmetic), so the pipe is busier than the flop rate
# says: `pipe_frac` counts instructions against the DFMA issue rate.
K1_FLOP_PER_PIXEL_ITER = 14.798e9 / (118326 * 16)           # 7816
K1_FP64_INSTR_PER_PIXEL_ITER = 9.725e9 / (118326 * 16)      # 5137
K1_FLOP_SOURCE = "profiles/r2_k1.txt"

# DRAM bytes per 4x4 block and CG iteration of cg_kernel, from the ncu --set
# full capture named below (dram__bytes_read.sum + dram__bytes_write.sum of a
# 200-iteration launch on the full system / (200 x its blocks)): H only, the
# preconditioner and the vectors stay in L2.
CG_DRAM_BYTES_PER_BLOCK_ITER = (26.721e9 + 0.250e9) / (200.0 * 1067206)   # 126.4
CG_TRAFFIC_SOURCE = "profiles/r2_cg.txt"


def cg_roofline(stats_sum, cg_ms, launches, hbm_peak, peak_source, views_per_launch=1):
    """Algorithmic bytes per CG iteration (DESIGN.md section 5): 128 per 4x4
    block of the system + per block row 128 (P) and 12 * 32 (vector passes).
    The system of a Newton step holds the blocks whose two nodes are still
    active (the reference drops the others, lib/gauss_newton_step.cc:91-105);
    the kernel reports their number."""
    cg_blocks, cg_rows = stats_sum
    algorithmic = cg_blocks * 128.0 + cg_rows * (128.0 + 12 * 32.0)
    achieved = (algorithmic / max(cg_ms * 1e-3, 1e-12)) / 1e9
    traffic = CG_DRAM_BYTES_PER_BLOCK_ITER * cg_blocks
    return {"bound": "hbm", "kernel": "cg_kernel (persistent PCG, one launch per Newton step"
            + (f", {views_per_launch} views per launch)" if views_per_launch > 1 else ")"),
            "achieved": achieved, "peak": hbm_peak, "peak_source": peak_source,
            "unit": "GB/s", "frac": achieved / hbm_peak,
            "traffic": traffic / max(launches, 1),
            "traffic_source": CG_TRAFFIC_SOURCE + ", scaled by system blocks x iterations",
            "frac_dram": traffic / max(cg_ms * 1e-3, 1e-12) / 1e9 / hbm_peak,
            "algorithmic_bytes_per_launch": algorithmic / max(launches, 1),
            "system_block_iterations_per_launch": cg_blocks / max(launches, 1),
            "launches_timed": launches}


def run_product(args):
    rank, world, local = dist_env()
    extras = not args.no_configs

    # ---- workloads first: forked builders must not inherit a CUDA context ----
    specs = [(WIDTH, HEIGHT, N_SUB, SCALE, False, s) for s in range(POOL)]
    if extras:
        specs += [(WIDTH, HEIGHT, N_SUB, SCALE, True, 100 + rank * BATCH + s)
                  for s in range(BATCH)]
    n_big = len(specs)
    want_cpu = (world == 1 and not args.no_cpu_baseline)
    if want_cpu:       # the CPU baselines' small views, built here too (no fork after CUDA)
        specs += [(SMALL_W, SMALL_H, N_SUB, SCALE, False, s) for s in range(4)]
        if extras:
            specs += [(SMALL_W, SMALL_H, N_SUB, SCALE, True, 100 + s) for s in range(2)]
    built = build_pool(specs)
    pool, pool_s = built[:POOL], built[POOL:n_big]
    small_n, small_s = built[n_big:n_big + 4], built[n_big + 4:]

    import torch
    import torch.distributed as dist
    from smvs_b200 import api

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (smvs_b200 has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def pin(a):
        # page-locked host copies: the e2e arm copies from pinned memory
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        return t.numpy()

    for wl in pool:
        wl.scene.images = [pin(a) for a in wl.scene.images]
        wl.nodes = pin(wl.nodes)
        wl.node_valid = pin(wl.node_valid)
        wl.patch_valid = pin(wl.patch_valid)
        wl.vis_off = pin(wl.vis_off)
        wl.vis_ids = pin(wl.vis_ids)
    # page-locked result buffers, one per context (the two-thread arm below
    # has two steps in flight)
    nodes_host = [pin(np.empty_like(wl.nodes)) for wl in pool]
    ctxs = [api.Context(local) for _ in pool]
    nodes_out = None
    e2e_parts = np.zeros(4)

    def view_of(step):
        return (rank + step) % POOL

    def e2e_step(step):
        j = view_of(step)
        wl, ctx = pool[j], ctxs[j]
        t = [time.perf_counter()]
        wl.push_views_u8(ctx)        # byte images; set_scale runs on the device
        t.append(time.perf_counter())
        wl.push_surface(ctx)
        t.append(time.perf_counter())
        st = ctx.newton_loop(None, REGULARIZATION, 0.0)
        t.append(time.perf_counter())
        nodes = ctx.get_nodes(out=nodes_host[j])
        t.append(time.perf_counter())
        e2e_parts[:] += np.diff(t)
        return st, nodes

    def resident_step(step):
        j = view_of(step)
        ctxs[j].set_nodes(pool[j].nodes)             # reset; not part of the timed loop
        return ctxs[j].newton_loop(None, REGULARIZATION, 0.0)

    sampler = ClockSampler(local)
    sampler.start()
    # warm-up (both paths, every view of the pool)
    for wl, ctx in zip(pool, ctxs):
        wl.push_views_u8(ctx)
        wl.push_surface(ctx)
    warm = max(args.warmup, 3)
    for s in range(max(warm, POOL)):
        resident_step(s)
    e2e_step(0)

    # ---- device-resident arm --------------------------------------------
    barrier()
    launches0 = sum(c.launches for c in ctxs)
    t_dev_ms, pix, newton, cg = 0.0, 0.0, 0, 0
    cg_blocks, cg_rows = 0.0, 0.0
    t_split = np.zeros(3)
    t0 = time.perf_counter()
    for s in range(args.steps):
        st = resident_step(s)
        t_dev_ms += st["ms_total"]
        pix += st["pixel_iterations"]
        newton += st["newton_steps"]
        cg += st["cg_iterations"]
        cg_blocks += st["cg_block_iterations"]
        cg_rows += st["cg_row_iterations"]
        t_split += [st["ms_construct"], st["ms_solve"], st["ms_update"]]
    barrier()
    t1 = time.perf_counter()
    wall_resident = t1 - t0
    launches = sum(c.launches for c in ctxs) - launches0
    clocks = sampler.stop(t0, t1)
    dump = {}
    if args.dump_outputs and args.steps > 0:
        last = ctxs[view_of(args.steps - 1)]
        dump["resident_nodes"] = last.get_nodes()
        dump["resident_depth"] = last.get_depth()
        dump["resident_stats"] = np.array([st[k] for k in DUMP_STATS], np.float64)

    # ---- end-to-end arm ---------------------------------------------------
    barrier()
    e2e_parts[:] = 0.0
    t0 = time.perf_counter()
    pix_e2e = 0.0
    for s in range(args.steps):
        st, nodes_out = e2e_step(s)
        pix_e2e += st["pixel_iterations"]
    barrier()
    wall_e2e = time.perf_counter() - t0
    if args.dump_outputs and args.steps > 0:
        dump["e2e_nodes"] = nodes_out.copy()

    # ---- end-to-end, two host threads per GPU ---------------------------------
    # The reference's host runs one view per pool thread (app/smvsrecon.cc:
    # 658-733) and the drop-in build gives thread k the device k mod N, so
    # with more pool threads than GPUs several views share a device: one
    # view's uploads and downloads overlap another's kernels. Same steps, same
    # copies per step; thread t takes the steps s = t (mod 2), which use
    # disjoint contexts (POOL is even). Reported next to the one-thread figure.
    import threading
    parts_1t = e2e_parts.copy()
    pix_2t = [0.0, 0.0]

    def e2e_worker(t):
        torch.cuda.set_device(local)
        for s in range(t, args.steps, 2):
            st, _ = e2e_step(s)
            pix_2t[t] += st["pixel_iterations"]

    barrier()
    t0 = time.perf_counter()
    workers2 = [threading.Thread(target=e2e_worker, args=(t,)) for t in range(2)]
    for th in workers2:
        th.start()
    for th in workers2:
        th.join()
    barrier()
    wall_e2e_2t = time.perf_counter() - t0
    pix_e2e_2t = sum(pix_2t)
    e2e_parts[:] = parts_1t

    # ---- reduce over ranks ---------------------------------------------------
    def reduce(vals_max, vals_sum):
        if world == 1:
            return list(vals_max), list(vals_sum)
        mx = torch.tensor(vals_max, dtype=torch.float64, device="cuda")
        sm = torch.tensor(vals_sum, dtype=torch.float64, device="cuda")
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        return mx.tolist(), sm.tolist()

    (t_dev_ms_max, wall_e2e_max, wall_e2e_2t_max), \
        (pix_all, pix_e2e_all, launches_all, pix_e2e_2t_all) = reduce(
            [t_dev_ms, wall_e2e, wall_e2e_2t],
            [pix, pix_e2e, float(launches), pix_e2e_2t])

    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_source = "MEASURED_PEAKS.json" if peaks else "fallback 6650 (B200_PROFILING.md)"

    configs = {}
    if extras:
        configs = run_extra_configs(args, api, torch, dist, rank, world, local, pool_s,
                                    ctxs, pin, barrier, reduce, hbm_peak, peak_source, small_s,
                                    dump)

    if rank == 0:
        value = pix_all / (t_dev_ms_max * 1e-3) / 1e6
        e2e_value = pix_e2e_all / wall_e2e_max / 1e6
        roofline = cg_roofline((cg_blocks, cg_rows), float(t_split[1]), newton, hbm_peak,
                               peak_source)
        roofline["system_blocks_full"] = _system_blocks_full(pool[0])
        # second roofline: the construct stage is fp64-ALU bound, not HBM bound
        roofline_k1 = None
        try:
            fp64_peak = api.measure_fp64_peak(local)
            k1_tflops = K1_FLOP_PER_PIXEL_ITER * pix / max(float(t_split[0]) * 1e-3, 1e-12) / 1e12
            roofline_k1 = {"bound": "fp64", "kernel": "gn_patch_kernel<16> (timed with the "
                           "assemble and preconditioner kernels of the construct stage)",
                           "achieved": k1_tflops, "peak": fp64_peak,
                           "peak_source": "smvsb_measure_fp64_peak (DFMA micro-benchmark, this run)",
                           "unit": "TFLOP/s", "frac": k1_tflops / fp64_peak,
                           "pipe_frac": k1_tflops * K1_FP64_INSTR_PER_PIXEL_ITER
                           / K1_FLOP_PER_PIXEL_ITER / (fp64_peak / 2.0),
                           "flop_per_pixel_iteration": K1_FLOP_PER_PIXEL_ITER,
                           "fp64_instructions_per_pixel_iteration": K1_FP64_INSTR_PER_PIXEL_ITER,
                           "flop_source": K1_FLOP_SOURCE}
        except Exception as exc:      # noqa: BLE001
            roofline_k1 = {"error": str(exc)}

        cpu_base = None          # timed on rank 0 at N = 1 only
        if not args.no_cpu_baseline and world == 1:
            try:
                workers = ReferenceWorkers(small_n, 4)
                p, s_ = workers.run_serial()
                workers.close()
                cpu_base = {"value": p / s_ / 1e6, "unit": UNIT, "cores": 1,
                            "kind": "reference",
                            "sample": "4 inner Newton loops, one after the other on one host "
                                      "thread: " + workers.desc}
            except Exception as exc:      # noqa: BLE001
                cpu_base = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference",
                            "sample": f"unavailable: {exc}"}

        config = dict(CONFIG)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": warm,
            "ms_per_step": t_dev_ms_max / max(args.steps, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config,
            "details": {"parallelism": f"views sharded, {world} GPU(s), no data-path collective",
                        "newton_steps_per_loop": newton / max(args.steps, 1),
                        "cg_iterations_per_loop": cg / max(args.steps, 1),
                        "mpix_iters_per_loop": pix / max(args.steps, 1) / 1e6,
                        "ms_construct_solve_update": [float(x) / max(args.steps, 1)
                                                      for x in t_split]},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT,
                    "h2d_bytes_per_step": pool[0].h2d_bytes_u8(),
                    "d2h_bytes_per_step": int(nodes_out.nbytes),
                    "ms_per_step": 1e3 * wall_e2e_max / max(args.steps, 1),
                    "ms_set_views_set_surface_loop_get_nodes":
                        [1e3 * float(x) / max(args.steps, 1) for x in e2e_parts],
                    "two_host_threads_per_gpu": {
                        "value": pix_e2e_2t_all / wall_e2e_2t_max / 1e6,
                        "ms_per_step": 1e3 * wall_e2e_2t_max / max(args.steps, 1),
                        "note": "same steps and copies, two views in flight per GPU "
                                "(one host thread each, like the reference's thread pool): "
                                "a view's copies overlap the other's kernels"}},
            "gpu_launches": int(launches_all),
            "roofline": roofline,
            "roofline_construct": roofline_k1,
            "cpu_baseline": cpu_base,
            "configs": configs,
            "wall_s_resident": wall_resident,
        }
        print(json.dumps(line))
        if args.dump_outputs:
            write_outputs(args.dump_outputs, dump)
    for c in ctxs:
        c.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_extra_configs(args, api, torch, dist, rank, world, local, pool_s, ctxs, pin,
                      barrier, reduce, hbm_peak, peak_source, small_s, dump):
    """BASELINE.json configs[2], [3], [4] -> the `configs` sub-dict."""
    out = {}
    steps = max(args.steps, 1)
    for wl in pool_s:
        wl.scene.images = [pin(a) for a in wl.scene.images]
    # the shading views re-use the contexts of the headline pool
    lights = []
    for wl, ctx in zip(pool_s, ctxs):
        wl.push_views_u8(ctx)
        wl.push_surface(ctx)
        lights.append(ctx.fit_lighting())          # lib/depth_optimizer.cc:110-117

    # ---- configs[2]: one view, -S ---------------------------------------
    def shading_step(j):
        ctxs[j].set_nodes(pool_s[j].nodes)
        return ctxs[j].newton_loop(lights[j], REGULARIZATION, 0.0)

    for j in range(len(pool_s)):
        shading_step(j)
    barrier()
    acc = dict(ms=0.0, pix=0.0, newton=0, cg=0, blocks=0.0, rows=0.0, split=np.zeros(3))
    for s in range(steps):
        st = shading_step((rank + s) % len(pool_s))
        acc["ms"] += st["ms_total"]
        acc["pix"] += st["pixel_iterations"]
        acc["newton"] += st["newton_steps"]
        acc["cg"] += st["cg_iterations"]
        acc["blocks"] += st["cg_block_iterations"]
        acc["rows"] += st["cg_row_iterations"]
        acc["split"] += [st["ms_construct"], st["ms_solve"], st["ms_update"]]
    barrier()
    if args.dump_outputs:
        dump["shading_nodes"] = ctxs[(rank + steps - 1) % len(pool_s)].get_nodes()
    (ms_max,), (pix_all,) = reduce([acc["ms"]], [acc["pix"]])
    if rank == 0:
        out["shading"] = {
            "workload": "configs[2]: 1 ref view + 6 neighbours, 1920x1080, scale 2, -S "
                        "(16 SH coefficients fitted per view, shading term on): inner Newton loop",
            "value": pix_all / (ms_max * 1e-3) / 1e6, "unit": UNIT, "steps": steps,
            "ms_per_step": ms_max / steps,
            "newton_steps_per_loop": acc["newton"] / steps,
            "cg_iterations_per_loop": acc["cg"] / steps,
            "ms_construct_solve_update": [float(x) / steps for x in acc["split"]],
            "roofline": cg_roofline((acc["blocks"], acc["rows"]), float(acc["split"][1]),
                                    acc["newton"], hbm_peak, peak_source)}

    # ---- configs[4]: BATCH views per GPU, -S ------------------------------
    # The views of a GPU advance in lock-step, `group` of them per PCG launch
    # (smvsb_newton_loop_batch): group = 1 is one view after the other, group
    # = BATCH all of them in one launch. Larger groups share the two grid-wide
    # synchronisations of a CG iteration but their vectors and preconditioners
    # (45 MB per view) no longer stay in the 126 MB L2 next to the Hessian
    # stream; every group size is measured, `value` is the best one.
    if hasattr(api, "newton_loop_batch"):
        nv = len(pool_s)

        def batch_step(group):
            for j in range(nv):
                ctxs[j].set_nodes(pool_s[j].nodes)
            sts = []
            for g0 in range(0, nv, group):
                sts += api.newton_loop_batch(ctxs[g0:g0 + group], lights[g0:g0 + group],
                                             REGULARIZATION, 0.0)
            return sts

        by_group = {}
        for group in sorted({1, 2, nv}):
            if group > nv:
                continue
            batch_step(group)
            barrier()
            acc = dict(ms=0.0, pix=0.0, blocks=0.0, rows=0.0, solve=0.0, launches=0)
            for s in range(steps):
                sts = batch_step(group)
                for g0 in range(0, nv, group):
                    acc["ms"] += sts[g0]["ms_total"]          # a group's device time
                    acc["solve"] += sts[g0]["ms_solve"]
                    acc["launches"] += max(st["newton_steps"] for st in sts[g0:g0 + group])
                for st in sts:
                    acc["pix"] += st["pixel_iterations"]
                    acc["blocks"] += st["cg_block_iterations"]
                    acc["rows"] += st["cg_row_iterations"]
            barrier()
            (ms_max,), (pix_all,) = reduce([acc["ms"]], [acc["pix"]])
            by_group[group] = dict(value=pix_all / (ms_max * 1e-3) / 1e6, ms_per_step=ms_max / steps,
                                   roofline=cg_roofline((acc["blocks"], acc["rows"]), acc["solve"],
                                                        acc["launches"], hbm_peak, peak_source,
                                                        views_per_launch=group))
        if rank == 0:
            best = max(by_group, key=lambda g: by_group[g]["value"])
            out["batch4"] = {
                "workload": f"configs[4]: {BATCH * world} ref views @ 2 MP, 6 neighbours each, "
                            f"-S, sharded over {world} GPU(s) ({BATCH} views/GPU, distinct "
                            "seeds); inner Newton loops of all views",
                "value": by_group[best]["value"], "unit": UNIT, "steps": steps,
                "ms_per_step": by_group[best]["ms_per_step"], "views_per_gpu": BATCH,
                "views_per_pcg_launch": best, "n_gpus": world, "scaling": "weak",
                "roofline": by_group[best]["roofline"],
                "by_views_per_launch": {str(g): {"value": v["value"], "ms_per_step": v["ms_per_step"],
                                                 "frac": v["roofline"]["frac"]}
                                        for g, v in by_group.items()}}

    # ---- configs[3]: SGM (rank 0, N = 1 only: it does not shard) -----------
    if world == 1:
        try:
            out["sgm"] = sgm_config(args, api, hbm_peak, peak_source, dump)
        except Exception as exc:      # noqa: BLE001
            out["sgm"] = {"error": str(exc)}

    # ---- CPU baselines of the extra configs (N = 1) -------------------------
    if world == 1 and rank == 0 and small_s and "shading" in out:
        try:
            workers = ReferenceWorkers(small_s, 2, shading=True)
            p, s_ = workers.run_serial()
            workers.close()
            out["shading"]["cpu_baseline"] = {
                "value": p / s_ / 1e6, "unit": UNIT, "cores": 1, "kind": "reference",
                "sample": "2 inner Newton loops, one after the other on one host thread: "
                          + workers.desc}
        except Exception as exc:      # noqa: BLE001
            out["shading"]["cpu_baseline"] = {"value": None, "sample": f"unavailable: {exc}"}
    return out


def sgm_config(args, api, hbm_peak, peak_source, dump):
    """configs[3]: SGM 1920x1080, 128 planes, P1 = 6, P2 = 96, 8 paths. Unit:
    Mvoxel/s (265.4 M voxels per run). Algorithmic bytes per voxel (SURVEY.md
    section 8d): 11 = cost write 1 + 8 path reads + final sum write 2."""
    from smvs_b200 import synth
    sc = synth.make_scene(WIDTH, HEIGHT, 1, seed_index=9)
    dmin, dmax = float(sc.true_depth.min() * 0.7), float(sc.true_depth.max() * 1.3)
    M, t = synth.reprojection(sc, 0)
    M, t = M.astype(np.float32), t.astype(np.float32)
    nvox = WIDTH * HEIGHT * 128
    for _ in range(3):
        r = api.sgm(sc.images[0], sc.images[1], M, t, dmin, dmax, 128)
    reps = max(args.steps, 1)
    ms = np.zeros(3)
    t0 = time.perf_counter()
    for _ in range(reps):
        r = api.sgm(sc.images[0], sc.images[1], M, t, dmin, dmax, 128)
        ms += r["ms"]
    wall = time.perf_counter() - t0
    ms /= reps
    if args.dump_outputs:
        dump["sgm_depth"] = r["depth"]
    dev_ms = float(ms.sum())
    out = {"workload": "configs[3]: sgm_stereo init, 1920x1080, 128 planes, 8-path aggregation "
                       "(cost volume + aggregation + WTA of one main/neighbour pair)",
           "value": nvox / (dev_ms * 1e-3) / 1e6, "unit": "Mvoxel/s", "runs": reps,
           "ms_per_run": dev_ms, "ms_cost_paths_wta": [float(x) for x in ms],
           "e2e": {"value": nvox / (wall / reps) / 1e6, "unit": "Mvoxel/s",
                   "h2d_bytes_per_step": 2 * WIDTH * HEIGHT,
                   "d2h_bytes_per_step": 4 * WIDTH * HEIGHT,
                   "ms_per_run": 1e3 * wall / reps},
           "valid_fraction": float((r["depth"] > 0).mean()),
           "roofline": {"bound": "hbm", "kernel": "SGM pipeline (cost + paths + sum/WTA)",
                        "achieved": 11.0 * nvox / (dev_ms * 1e-3) / 1e9, "peak": hbm_peak,
                        "peak_source": peak_source, "unit": "GB/s",
                        "frac": 11.0 * nvox / (dev_ms * 1e-3) / 1e9 / hbm_peak,
                        "algorithmic_bytes_per_voxel": 11}}
    if not args.no_cpu_baseline:
        try:
            from oracle import ref as oref
            small = synth.make_scene(SMALL_W, SMALL_H, 1, seed_index=9)
            R = oref.RefScene(small)
            t0 = time.perf_counter()
            R.sgm_run(0, 1, 0, 128, dmin, dmax)
            secs = time.perf_counter() - t0
            R.close()
            out["cpu_baseline"] = {
                "value": SMALL_W * SMALL_H * 128 / secs / 1e6, "unit": "Mvoxel/s", "cores": 1,
                "kind": "reference",
                "sample": f"SGMStereo::run_sgm on one {SMALL_W}x{SMALL_H} pair, 128 planes "
                          "(1/16 of the voxels), one host thread"}
        except Exception as exc:      # noqa: BLE001
            out["cpu_baseline"] = {"value": None, "sample": f"unavailable: {exc}"}
    return out


def write_outputs(path, arrays):
    """DIR/<name>.npy of each output, float32 / float64 as computed."""
    os.makedirs(path, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"bench.py: outputs of {total} bytes exceed {DUMP_LIMIT}")
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(path, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="smvs_b200", choices=["smvs_b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true",
                    help="skip the `configs` sub-dict (BASELINE.json configs[2..4])")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step of each timed "
                         "path returned to DIR/<name>.npy: resident_nodes / resident_depth / "
                         "resident_stats (headline loop), e2e_nodes, and with the configs "
                         "shading_nodes and sgm_depth; the inputs are seeded, so two builds "
                         "can be compared output for output")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    return run_product(args)


if __name__ == "__main__":
    sys.exit(main())
