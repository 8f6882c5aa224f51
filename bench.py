#!/usr/bin/env python
"""bench.py -- headline benchmark of the render hot path (BASELINE.json: path samples/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload C3]

One "step" = one pass of the path tracer over the whole frame: `spp` samples for every pixel of the
workload (default C3, the configuration the metric is quoted on: 512^3 u16 volume, 1920x1080, Woodcock
tracking, single scattering, area + environment light, 256 spp), accumulated into a float4 sum buffer,
reduced over the ranks (N > 1: one NCCL sum-reduce of the per-GPU buffers onto rank 0) and resolved
(divide + tone map) into the u8 image.  Weak scaling: every rank renders `spp` samples of its own; like a progressive
render the sample range advances with every step (step g, rank r: sample indices [(g*N + r)*spp, (g*N + r + 1)*spp)),
so no step replays the taps of the one before.  N > 1 also reports the STRONG split (the workload's spp divided over
the ranks, reduce + resolve inside the timed region) and, with enough GPUs and memory, C5.

  value     whole-job samples/s with the scene resident in HBM, CUDA events over exactly K steps,
            max over ranks.
  e2e       the same through the C ABI from HOST buffers: every step uploads the voxels from pinned
            host memory into the volume's cudaArray (which invalidates and rebuilds the macrocell grid;
            N > 1: one PCIe upload on rank 0 + an NCCL broadcast over NVLink), re-uploads the
            transfer-function table, re-publishes camera and lights, renders, and reads the tone-mapped
            image and the float accumulator back into pinned host memory.  Frames are streamed: the
            upload of step i+1 runs on a copy stream beside the rendering of step i (render.VolumeStream)
            and the read-back of step i beside the binding and rendering of step i+1; the same loop
            without any overlap is reported as e2e.ms_per_step_without_overlap.
  roofline  nominal HBM figure: algorithmic bytes per launch (COUNTED taps x 8 voxels x bytes/voxel + TF lookups x 32 B
            + framebuffer bytes, SURVEY.md section 8d) / the path-tracing kernel's mean launch duration
            measured with CUDA events inside the timed region, against MEASURED_PEAKS.json; `gather`: the kernel's
            taps/s against the tex3D ceilings measured here on the benched volume (coherent and random taps, the
            metric's "% of gather roofline"); `issue`: issue-slot utilisation and lanes per instruction of the
            same kernel from the committed ncu capture -- the bound that actually limits it.
  cpu_baseline  the CPU oracle (port of the reference's device code, OpenMP over rows) on a bounded
            sample of the same workload -- test infrastructure used as a yardstick, never the product.

--impl reference: the reference has no CPU render path (SURVEY.md section 8c); its implementation of
this path IS its CUDA kernels.  The arm runs them unmodified (oracle/_ref, compiled from
/root/reference by oracle/Makefile) on one B200 through the reference's own entry points and frame
protocol (render_pathtracer once per sample, three launches each).  Its scene (cudaArray, texture objects,
synthetic voxels) is built by oracle/ref_scene.cu with plain CUDA runtime calls: the arm's process never loads
libsvr_b200.so.  `--ref-device cpu` times the CPU port instead.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "path_samples_per_sec"
UNIT = "samples/s"


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# clocks sampled DURING the timed regions (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        import torch

        self.path = tempfile.mktemp(prefix="svr_clocks_", suffix=".csv")
        self.proc = None
        self.windows = []
        try:
            uuid = str(torch.cuda.get_device_properties(device_index).uuid)
            ident = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
        except Exception:
            ident = str(device_index)
        try:
            self.out = open(self.path, "w")
            self.proc = subprocess.Popen(
                ["nvidia-smi", "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits", "-lms", "100", "-i", ident],
                stdout=self.out, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def window(self, t0, t1):
        self.windows.append((t0, t1))

    def finish(self):
        import datetime

        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()  # the exact process we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.out.close()
        rows = []
        try:
            with open(self.path) as f:
                for line in f:
                    p = [x.strip() for x in line.split(",")]
                    if len(p) < 8:
                        continue
                    try:
                        ts = datetime.datetime.strptime(p[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                        rows.append((ts, float(p[1]), float(p[2]), float(p[3]), p[4:8]))
                    except ValueError:
                        continue
            os.unlink(self.path)
        except OSError:
            pass
        inside = [r for r in rows if any(t0 - 0.05 <= r[0] <= t1 + 0.05 for t0, t1 in self.windows)]
        used = inside if inside else rows
        if not used:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in used for i in range(4) if r[4][i].lower().startswith("active")})
        return {
            "sm_mhz": statistics.median(r[1] for r in used),
            "sm_max_mhz": max(r[2] for r in used),
            "power_w_max": max(r[3] for r in used),
            "samples": len(used),
            "samples_in_timed_region": len(inside),
            "reasons": reasons,
        }


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def algorithmic_bytes(cnt, voxel_bytes, npix, passes=1):
    """SURVEY.md section 8(d): taps x 8 voxels x B_v + TF lookups x 32 B + framebuffer bytes (one float4
    read-modify-write of the accumulator per launch)."""
    taps = cnt["track_taps"] + cnt["shadow_taps"] + cnt["shade_taps"]
    return taps * 8 * voxel_bytes + cnt["tf_lookups"] * 32 + passes * npix * 32, taps


def grid_cell(r):
    """Edge, in voxels, of the macrocell grid the library built for the scene (chosen automatically unless --cell)."""
    dims, cell = (C.c_int32 * 3)(), C.c_int32()
    if r.lib.svr_grid_info(dims, C.byref(cell)) != 0:
        return None
    return int(cell.value)



def gather_ceilings(r, achieved_gtaps=None):
    """The metric's "% of gather roofline": the texture unit's tap rate on the BENCHED volume, measured here with
    dependence-free tex3D loops (svr_microbench_taps) -- coherent (neighbouring lanes walk neighbouring rays: the best the
    unit does) and random (hashed coordinates over the whole volume: every tap a miss) -- and the path tracer's counted
    taps per second as a fraction of each.  Best of 3 launches."""
    import torch

    from sunvolumerender_b200 import _lib as L

    out = {}
    sink = torch.zeros(4, dtype=torch.float32, device="cuda")
    for name, rnd, threads, per in (("coherent", 0, 1 << 20, 512), ("random", 1, 1 << 20, 128)):
        taps_out = C.c_uint64(0)
        best = None
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            L.check(r.lib.svr_microbench_taps(C.byref(r.volume), rnd, threads, per, C.c_void_p(sink.data_ptr()), C.byref(taps_out)))
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None else min(best, ms)
        g = taps_out.value / (best * 1e-3) / 1e9
        out[f"{name}_gtaps_per_s"] = round(g, 2)
    out["peak_source"] = "measured here: 2^20 threads x 512 coherent / 128 random tex3D taps on the benched volume, best of 3"
    return out


def layout_study(r, voxels16, n):
    """north_star offers "a bricked, Morton-ordered layout bound as a 3D texture object or staged through shared memory" for
    the voxels; the product keeps the caller's cudaArray texture (hardware block-linear tiling, filter in the texture unit).
    The measurement behind that: the same independent trilinear taps -- coherent and random -- (0) as one TEX on the
    cudaArray, (1) in software from a linear copy (8 loads + filter in the SM), (2) in software from a copy in 8^3-voxel
    bricks in Morton order.  `voxels16`: the volume's n^3 16-bit voxels on the device.  G taps/s, best of 3."""
    import torch

    from sunvolumerender_b200 import _lib as L

    sink = torch.zeros(4, dtype=torch.float32, device="cuda")
    bricked = torch.empty_like(voxels16)
    L.check(r.lib.svr_layout_brick(C.c_void_p(voxels16.data_ptr()), C.c_void_p(bricked.data_ptr()), n))
    torch.cuda.synchronize()

    def rate(launch):
        taps_out, best = C.c_uint64(0), None
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            launch(taps_out)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None else min(best, ms)
        return round(taps_out.value / (best * 1e-3) / 1e9, 2)

    out = {}
    for name, rnd, per in (("coherent", 0, 256), ("random", 1, 64)):
        out[name] = {
            "cudaarray_tex3d": rate(lambda t: L.check(r.lib.svr_microbench_taps(C.byref(r.volume), rnd, 1 << 20, per, C.c_void_p(sink.data_ptr()), C.byref(t)))),
            "linear_software_trilinear": rate(lambda t: L.check(r.lib.svr_microbench_soft_taps(C.c_void_p(voxels16.data_ptr()), n, 1, rnd, 1 << 20, per, C.c_void_p(sink.data_ptr()), C.byref(t)))),
            "bricked_morton_software_trilinear": rate(lambda t: L.check(r.lib.svr_microbench_soft_taps(C.c_void_p(bricked.data_ptr()), n, 2, rnd, 1 << 20, per, C.c_void_p(sink.data_ptr()), C.byref(t)))),
        }
    out["unit"] = "G taps/s (2^20 threads x 256 coherent / 64 random independent trilinear taps, best of 3)"
    return out


def issue_counters(workload, spp, kernel):
    """Issue-slot utilisation and lanes per instruction of the dominant kernel, from the committed ncu --set full capture of
    this very launch (profiles/r02/issue.json, written by tools/ncu_issue.py from the .ncu-rep): the bound that limits it."""
    for rnd in ("r02", "r01"):
        path = os.path.join(ROOT, "profiles", rnd, "issue.json")
        try:
            with open(path) as f:
                for e in json.load(f):
                    if e.get("workload") == workload and e.get("spp") == spp and e.get("kernel") == kernel:
                        return dict(e, source=f"profiles/{rnd}/issue.json")
        except Exception:
            continue
    return None


def timed_steps(fn, steps, warmup, barrier, dev):
    """`steps` calls of fn() after `warmup`, CUDA events, max over ranks -> ms per step."""
    import torch

    from sunvolumerender_b200 import distributed as D

    for _ in range(warmup):
        fn()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    barrier()
    return D.max_over_ranks(e0.elapsed_time(e1), dev) / steps


def strong_scaling_line(r, a, cfg, sum_buf, rank, world, dev, barrier):
    """north_star's multi-GPU split of ONE frame (C3: 256 spp per pixel in all), everything inside the timed region, two ways:
      samples  the spp divided over the GPUs (256 / N each), one NCCL sum-reduce of the float4 accumulators onto rank 0,
               resolve there;
      bands    the IMAGE divided: row bands dealt out round robin, every GPU renders all 256 spp of its pixels straight into
               rank 0's accumulator through peer mappings over NVLink (svr_pathtracer_accumulate_bands + distributed.PeerFrame:
               no collective), rank 0 resolves.  Per-pixel set-up is divided as well, and the frame is bit-identical to the
               single-GPU frame (checked here).
    The speed-up over one GPU is computed by whoever reads the N = 1 line."""
    import torch
    import torch.distributed as dist

    from sunvolumerender_b200 import _lib as L
    from sunvolumerender_b200 import distributed as D
    from sunvolumerender_b200 import scene as S

    spp = a.spp or cfg.spp
    parts = S.split_samples(spp, world)
    first, count = parts[rank]
    npix = cfg.width * cfg.height
    g = [0]

    def step(render=True, reduce=True):
        base = g[0] * spp
        g[0] += 1
        if render and count:
            r.accumulate(sum_buf, cfg.trace_depth, base + first, count, clear=True)
        elif render:
            sum_buf.zero_()
        if reduce:
            dist.reduce(sum_buf, dst=0, op=dist.ReduceOp.SUM)
            if rank == 0:
                r.resolve(sum_buf)

    ms = timed_steps(step, a.steps, max(a.warmup, 3), barrier, dev)
    ms_render = timed_steps(lambda: step(True, False), max(3, a.steps // 2), 1, barrier, dev)
    ms_reduce = timed_steps(lambda: step(False, True), max(3, a.steps // 2), 1, barrier, dev)
    line = {"workload": f"{cfg.name}: ONE frame of {spp} spp on {world} GPUs, device-resident, assembly and resolve on rank 0 inside the timed region",
            "scaling": "strong", "unit": UNIT, "spp_total": spp,
            "split_samples": {"value": npix * spp / (ms * 1e-3), "ms_per_step": ms, "spp_per_gpu": count, "ms_render_only": ms_render,
                              "ms_reduce_and_resolve_only": ms_reduce, "exchange": f"NCCL sum-reduce of {npix * 16 / 1e6:.1f} MB float4 accumulators",
                              "limiter": "the per-pixel accumulator pass is paid by every GPU for every pixel, and 32-sample launches leave a warp one round per pixel (it waits for its longest path): render time does not shrink like 1/N"}}
    try:
        pf = D.PeerFrame(r, npix * 16)
        gb = [0]

        def step_bands():
            base = gb[0] * spp
            gb[0] += 1
            r.accumulate_bands(pf.img_ptr, cfg.trace_depth, base, spp, rank, world, clear=True)
            pf.frame_done()
            if rank == 0:
                r.resolve(pf.img_ptr)
            dist.barrier()  # the next frame goes into the same buffer (a real host would double-buffer; the barrier is timed)

        ms_b = timed_steps(step_bands, a.steps, max(a.warmup, 3), barrier, dev)
        # With few pixels per GPU the frame ends when the last block does: shorter blocks shorten that tail -- runs of 1 pixel
        # per warp, and / or the warps of a block splitting the samples of one row's pixels (SVR_OPT_PT_BLOCK_SPLIT).
        wp0 = r.get_option(L.OPT_PT_WARP_PIXELS)   # 0 = the library's choice by launch length
        best_cfg = (wp0, 0)
        if world >= 4:
            for cand in dict.fromkeys(c for c in ((1, 0), (2, 0), (wp0, 1), (1, 1)) if c != (wp0, 0)):
                r.set_option(L.OPT_PT_WARP_PIXELS, cand[0])
                r.set_option(L.OPT_PT_BLOCK_SPLIT, cand[1])
                ms_c = timed_steps(step_bands, a.steps, 2, barrier, dev)
                if ms_c < ms_b:
                    ms_b, best_cfg = ms_c, cand
            r.set_option(L.OPT_PT_WARP_PIXELS, best_cfg[0])
            r.set_option(L.OPT_PT_BLOCK_SPLIT, best_cfg[1])
            step_bands()   # the last frame (checked below) is rendered with the setting that is reported
        same = None
        if rank == 0:   # the last frame against the same samples on one GPU
            assembled = r.hdr.clone()
            r.accumulate(sum_buf, cfg.trace_depth, (gb[0] - 1) * spp, spp, clear=True)
            r.resolve(sum_buf)
            torch.cuda.synchronize()
            same = bool(torch.equal(assembled, r.hdr))
        barrier()
        pf.close()
        r.set_option(L.OPT_PT_WARP_PIXELS, wp0)
        r.set_option(L.OPT_PT_BLOCK_SPLIT, 0)
        line["split_bands"] = {"value": npix * spp / (ms_b * 1e-3), "ms_per_step": ms_b, "pixels_per_warp_run": best_cfg[0], "block_split": best_cfg[1], "exchange": "peer writes into rank 0's accumulator, completion flags, no collective "
                               "(+ one barrier per frame, timed, because frames share the buffer)", "equals_single_gpu_frame": same}
    except Exception as e:  # no peer access between these GPUs
        line["split_bands"] = {"unavailable": str(e)}
    best = max((v for v in (line["split_samples"], line["split_bands"]) if "value" in v), key=lambda v: v["value"])
    line["value"], line["ms_per_step"] = best["value"], best["ms_per_step"]
    line["split"] = "bands" if best is line["split_bands"] else "samples"
    return line


def c5_line(r, a, rank, world, dev, barrier):
    """BASELINE.json configs[4]: 2048^3 u16 (16 GiB, replicated on every GPU), 3840x2160, 1024 spp split across the GPUs of the
    box with one NCCL reduce of the accumulation buffers; and the same frame with the image split instead (row bands, peer
    writes, see strong_scaling_line).  Run when the box has 8 GPUs (or --c5) and the memory for it."""
    import torch
    import torch.distributed as dist

    from sunvolumerender_b200 import distributed as D
    from sunvolumerender_b200 import scene as S
    from sunvolumerender_b200.render import setup_config

    if world < 8 and not a.c5:
        return None
    cfg = S.CONFIGS["C5"]
    free, _ = torch.cuda.mem_get_info(dev)
    ok = torch.tensor([1 if free > 44 * 2 ** 30 else 0], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if int(ok.item()) == 0:
        return {"workload": "C5", "unavailable": "needs ~40 GiB of free device memory per GPU (16 GiB of voxels + the generator's buffer)"}
    vb = setup_config(r, cfg)
    del vb
    torch.cuda.empty_cache()
    W, H, spp = cfg.width, cfg.height, cfg.spp
    first, count = S.split_samples(spp, world)[rank]
    buf = torch.zeros(W * H * 4, dtype=torch.float32, device=dev)
    g = [0]

    def step():
        base = g[0] * spp
        g[0] += 1
        r.accumulate(buf, cfg.trace_depth, base + first, count, clear=True)
        dist.reduce(buf, dst=0, op=dist.ReduceOp.SUM)
        if rank == 0:
            r.resolve(buf)

    ms = timed_steps(step, 3, 2, barrier, dev)
    nz = float((r.ldr_image()[..., :3] > 0).float().mean()) if rank == 0 else None
    line = {"workload": f"C5: 2048^3 u16 (16 GiB replicated), {W}x{H}, ONE frame of {spp} spp on {world} GPUs, device-resident, assembly + resolve on rank 0 inside "
                        f"the timed region, 3 steps",
            "scaling": "strong", "unit": UNIT, "macrocell": grid_cell(r), "image_nonzero_fraction": nz,
            "split_samples": {"value": W * H * spp / (ms * 1e-3), "ms_per_step": ms, "spp_per_gpu": count, "exchange": f"NCCL sum-reduce of {W * H * 16 / 1e6:.0f} MB accumulators"}}
    try:
        pf = D.PeerFrame(r, W * H * 16)
        gb = [0]

        def step_bands():
            base = gb[0] * spp
            gb[0] += 1
            r.accumulate_bands(pf.img_ptr, cfg.trace_depth, base, spp, rank, world, clear=True)
            pf.frame_done()
            if rank == 0:
                r.resolve(pf.img_ptr)
            dist.barrier()

        ms_b = timed_steps(step_bands, 3, 2, barrier, dev)
        pf.close()
        line["split_bands"] = {"value": W * H * spp / (ms_b * 1e-3), "ms_per_step": ms_b, "exchange": "peer writes into rank 0's accumulator, completion flags, one barrier per frame"}
    except Exception as e:
        line["split_bands"] = {"unavailable": str(e)}
    best = max((v for v in (line["split_samples"], line["split_bands"]) if "value" in v), key=lambda v: v["value"])
    line["value"], line["ms_per_step"] = best["value"], best["ms_per_step"]
    line["split"] = "bands" if best is line["split_bands"] else "samples"
    del buf
    setup_config(r, S.CONFIGS["C1"])  # drop the 16 GiB array
    torch.cuda.empty_cache()
    return line


def run_ours(a):
    import numpy as np
    import torch
    import torch.distributed as dist

    from sunvolumerender_b200 import _lib as L
    from sunvolumerender_b200 import distributed as D
    from sunvolumerender_b200 import scene as S
    from sunvolumerender_b200.render import Renderer, setup_config

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # rank 0 prints ONE JSON line on stdout: keep NCCL's own banner ("NCCL version ...") out of it
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    cfg = S.CONFIGS[a.workload]
    spp = a.spp or cfg.spp
    depth = cfg.trace_depth
    W, H = cfg.width, cfg.height
    npix = W * H

    r = Renderer(local)
    vb = setup_config(r, cfg)  # synthetic voxels generated on the device (svr_generate_volume)
    r.set_option(L.OPT_PT_MODE, a.pt_mode)
    if os.environ.get("SVR_BENCH_FUSED_UPLOAD") == "0":  # A/B of the e2e leg: copy + range kernel instead of the one-pass upload
        r.set_option(L.OPT_FUSED_UPLOAD, 0)
    if a.cell:
        r.set_option(L.OPT_MACROCELL_SIZE, a.cell)
    sum_buf = torch.zeros(npix * 4, dtype=torch.float32, device=dev)
    gstep = [0]  # steps rendered so far: like a progressive render, every step takes the next sample range

    def next_first(n_spp=None):
        n_spp = spp if n_spp is None else n_spp
        first = (gstep[0] * world + rank) * n_spp
        gstep[0] += 1
        return first

    def render_step(time_kernel=None):
        first = next_first()
        if time_kernel is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        r.accumulate(sum_buf, depth, first, spp, clear=True)
        if time_kernel is not None:
            e1.record()
            time_kernel.append((e0, e1))
        if world > 1:
            dist.reduce(sum_buf, dst=0, op=dist.ReduceOp.SUM)
        if rank == 0:
            r.resolve(sum_buf)

    # ---- counted taps of one launch (the sample range of this rank's first step; the counts of later ranges differ by
    # Monte Carlo noise, a few 1e-4 relative)
    r.set_option(L.OPT_COUNTERS, 1)
    r.reset_counters()
    r.accumulate(sum_buf, depth, rank * spp, spp, clear=True)
    torch.cuda.synchronize()
    cnt = r.counters()
    r.set_option(L.OPT_COUNTERS, 0)

    clocks = ClockSampler(local) if rank == 0 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: scene resident in HBM
    for _ in range(a.warmup):
        render_step()
    barrier()
    launches0 = r.launch_count()
    kernel_events = []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    ev0.record()
    for _ in range(a.steps):
        render_step(kernel_events)
    ev1.record()
    barrier()
    t1 = time.time()
    ms_local = ev0.elapsed_time(ev1)
    launches = r.launch_count() - launches0
    if clocks:
        clocks.window(t0, t1)
    ms = D.max_over_ranks(ms_local, dev)
    kernel_ms = sum(x.elapsed_time(y) for x, y in kernel_events) / len(kernel_events)
    value = npix * spp * world * a.steps / (ms * 1e-3)
    if a.dump_outputs and rank == 0:  # the last timed step's images, before the legs below render into the same buffers
        dump_outputs(a.dump_outputs, {"hdr": r.hdr_image(), "ldr": r.ldr_image()})
    cell_used = grid_cell(r)  # before other scenes are loaded into the renderer
    base_volume, base_camera, base_lights = r.volume, r.camera, list(r.lights)  # the PODs of the benched scene (copies are taken by the oracle)
    gather = gather_ceilings(r) if rank == 0 else None

    # ---- e2e: everything from host buffers, results back on the host
    def run_e2e():
        host_vox = torch.empty(vb.numel(), dtype=torch.uint8, pin_memory=True)
        host_vox.copy_(vb)
        host_img = torch.empty(npix * 4, dtype=torch.uint8, pin_memory=True)
        host_hdr = torch.empty(npix * 3, dtype=torch.float32, pin_memory=True)
        tf_table = S.tf_table(cfg.tf)
        cam = S.default_camera(cfg.extent, W, H)
        lights = [S.default_area_light(cfg.extent)]
        env = S.constant_env_light()
        torch.cuda.synchronize()

        # Frames stream through the renderer the way a time series of volumes would: while frame i renders, the
        # voxels of frame i+1 cross PCIe on a copy stream into a staging buffer (render.VolumeStream); N > 1: they
        # cross PCIe ONCE (rank 0) and reach the other GPUs over NVLink -- pushed by copy engines into peer-mapped
        # staging buffers ("p2p"), or with an NCCL broadcast ("nvlink") -- instead of N uploads competing for host
        # memory bandwidth ("pcie").  Every step still uploads its own inputs and reads its own results back
        # inside the timed region: K prefetches, K binds, K read-backs for K steps.
        from sunvolumerender_b200.render import VolumeStream

        bgroup = None
        if world > 1 and a.e2e_fanout == "nvlink":
            opts = dist.ProcessGroupNCCL.Options()
            opts.is_high_priority_stream = True
            bgroup = dist.new_group(pg_options=opts)  # the broadcast gets its own communicator and stream
        vs = VolumeStream(r, vb.numel(), group=bgroup, fanout=a.e2e_fanout)
        fanout = vs.fanout

        # Results stream out the same way: rank 0 resolves frame i, a read-back stream copies image + accumulator to
        # pinned host buffers (double-buffered) while frame i+1 is being bound and rendered, and the caller looks
        # at frame i-1.  The setup_* calls of the next frame must not wait for that copy: SVR_OPT_SETUP_SYNC = 0.
        rb_stream = torch.cuda.Stream(device=dev)
        host_imgs = [host_img, torch.empty_like(host_img).pin_memory()]
        host_hdrs = [host_hdr, torch.empty_like(host_hdr).pin_memory()]
        resolved = [torch.cuda.Event(), torch.cuda.Event()]
        read_back = [torch.cuda.Event(), torch.cuda.Event()]

        h2d_trace = []
        trace = [] if os.environ.get("SVR_BENCH_E2E_TRACE") else None  # per-step events on the render stream (stderr, diagnostic)

        def mark(row):
            if trace is not None:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                row.append(e)

        def e2e_step(i, prefetch_next, serial=False):
            main = torch.cuda.current_stream()
            row = []
            if trace is not None and not serial:
                trace.append(row)
            mark(row)
            if serial:
                vs.prefetch(host_vox)                  # no overlap: transfer, then render
            vs.bind()                                  # staged voxels -> cudaArray; macrocell ranges rebuilt at the next render
            mark(row)
            r.set_transfer_function(tf_table)          # H2D 16 KiB table into the bound 1-D array
            r.set_camera(cam)
            r.set_area_lights(lights)
            r.set_env_light(env, enabled=cfg.env)
            r.accumulate(sum_buf, depth, next_first(), spp, clear=True)
            mark(row)
            if prefetch_next and not serial:
                if trace is not None:
                    h0 = torch.cuda.Event(enable_timing=True)
                    h0.record(vs.copy_stream)
                vs.prefetch(host_vox)                  # H2D (+ fan-out) of the NEXT frame, beside this frame's render kernel
                if trace is not None:
                    h1 = torch.cuda.Event(enable_timing=True)
                    h1.record(vs.copy_stream)
                    h2d_trace.append((row, h0, h1))
            if rank == 0 and not serial and i > 0:
                issue_read_back((i - 1) & 1)           # frame i-1 leaves for the host while frame i renders ...
                read_back[(i - 1) & 1].synchronize()   # ... and the caller looks at it
            if world > 1:
                dist.reduce(sum_buf, dst=0, op=dist.ReduceOp.SUM)
            if rank == 0:
                slot = i & 1
                main.wait_event(read_back[slot ^ 1])   # resolve overwrites r.img / r.hdr: the previous frame's copy has left
                r.resolve(sum_buf)
                mark(row)
                if serial:
                    host_imgs[slot].copy_(r.img, non_blocking=True)
                    host_hdrs[slot].copy_(r.hdr, non_blocking=True)
                    main.synchronize()                 # the caller looks at this frame
                else:
                    resolved[slot].record(main)

        def issue_read_back(slot):
            # A bulk device-to-host copy that starts between two frames delays the kernels that refresh the next frame's volume
            # and grid (measured: +0.35 ms on a 0.25 ms upload kernel), a render kernel does not notice it: so frame i-1 is read
            # back once frame i's render kernel has been launched.
            with torch.cuda.stream(rb_stream):
                rb_stream.wait_event(resolved[slot])
                host_imgs[slot].copy_(r.img, non_blocking=True)
                host_hdrs[slot].copy_(r.hdr, non_blocking=True)
                read_back[slot].record(rb_stream)

        def e2e_run(steps, serial):
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            r.set_option(L.OPT_SETUP_SYNC, 1 if serial else 0)
            barrier()
            t0 = time.time()
            ev0.record()
            if not serial:
                vs.prefetch(host_vox)
            for i in range(steps):
                e2e_step(i, i + 1 < steps, serial)
            if rank == 0 and not serial:
                issue_read_back((steps - 1) & 1)
                read_back[(steps - 1) & 1].synchronize()   # the last frame has reached the host
            ev1.record()
            barrier()
            t1 = time.time()
            r.set_option(L.OPT_SETUP_SYNC, 1)
            return D.max_over_ranks(ev0.elapsed_time(ev1), dev), (t0, t1)

        e2e_run(max(1, min(a.warmup, 2)), False)
        e2e_serial_ms, _ = e2e_run(max(2, a.steps // 4), True)
        e2e_serial_ms /= max(2, a.steps // 4)
        e2e_ms, win = e2e_run(a.steps, False)
        if clocks:
            clocks.window(*win)
        e2e_value = npix * spp * world * a.steps / (e2e_ms * 1e-3)
        if trace and rank == 0:
            rows = [t for t in trace[-a.steps:] if len(t) == 4]
            seg = [sum(t[k].elapsed_time(t[k + 1]) for t in rows) / len(rows) for k in range(3)]
            gap = sum(rows[k][3].elapsed_time(rows[k + 1][0]) for k in range(len(rows) - 1)) / max(1, len(rows) - 1)
            hh = [(h0.elapsed_time(h1), rw[1].elapsed_time(h0), rw[1].elapsed_time(h1), rw[1].elapsed_time(rw[2])) for rw, h0, h1 in h2d_trace[-(a.steps - 1):] if len(rw) == 4]
            if hh:
                print("e2e trace (ms): next frame's H2D takes %.3f; relative to the end of bind it starts at %.3f and ends at %.3f, the render ends at %.3f"
                      % tuple(sum(x[k] for x in hh) / len(hh) for k in range(4)), file=sys.stderr)
            print("e2e trace (ms): bind per step " + " ".join("%.2f" % t[0].elapsed_time(t[1]) for t in rows), file=sys.stderr)
            print(f"e2e trace (ms, render stream): bind {seg[0]:.3f}  grid build + render {seg[1]:.3f}  reduce + resolve {seg[2]:.3f}  "
                  f"between steps {gap:.3f}  (device-resident render {kernel_ms:.3f})", file=sys.stderr)
        small = tf_table.nbytes + 112 + 16 + 76 + 44 * len(lights) + 32  # table + scene PODs, every rank
        h2d = int(vb.numel() * (world if fanout == "pcie" else 1) + small * world)
        d2h = int(host_img.numel() + host_hdr.numel() * 4)
        last = host_imgs[(a.steps - 1) & 1]
        img_nonzero = float((last.view(H, W, 4)[..., :3] > 0).float().mean()) if rank == 0 else 0.0
        if rank == 0:  # what reached the host is the frame on the device
            assert torch.equal(last, r.img.cpu()) and torch.equal(host_hdrs[(a.steps - 1) & 1], r.hdr.cpu()), "e2e read-back differs from the device image"
        vs.close()
        return {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / a.steps,
                "pipeline": "frame i+1's H2D and frame i-1's D2H overlap frame i's render (VolumeStream, read-back stream); every step uploads and reads back",
                "ms_per_step_without_overlap": e2e_serial_ms, "fanout": fanout}, img_nonzero

    if a.no_e2e or (vb.numel() > (2 << 30) and not a.force_e2e):
        # a 16 GiB volume per rank would pin 16 GiB of host memory per rank: opt in with --force-e2e
        e2e, img_nonzero = None, None
    else:
        e2e, img_nonzero = run_e2e()

    # ---- N > 1: the STRONG split north_star states (the workload's spp divided over the GPUs, one NCCL sum-reduce of
    # the float4 accumulators, resolve on rank 0 -- all inside the timed region), and C5 where it fits
    strong = strong_scaling_line(r, a, cfg, sum_buf, rank, world, dev, barrier) if world > 1 else None
    c5 = c5_line(r, a, rank, world, dev, barrier) if world > 1 and not a.no_c5 else None

    # the metric's second half at N > 1 (collective: every rank takes part)
    raycast_multi = raycast_lines_multi(r, rank, world, dev) if world > 1 and not a.no_raycast else None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    clk = clocks.finish()

    # ---- roofline of the dominant kernel (the path-tracing launch)
    peak, peak_src = measured_peak()
    bytes_algo, taps = algorithmic_bytes(cnt, cfg.voxel_bytes, npix)
    achieved = bytes_algo / (kernel_ms * 1e-3) / 1e9
    warp_shape = r.get_option(L.OPT_PT_KERNEL) == 2 and spp >= r.get_option(L.OPT_PT_WARP_MIN_SPP)
    roofline_kernel = f"pathtrace_{'warp' if warp_shape else 'mega'}_kernel<{a.pt_mode},0>"
    traffic = None  # dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed ncu --set full capture
    try:
        for rnd in ("r02", "r01"):
            path = os.path.join(ROOT, "profiles", rnd, "traffic.json")
            if not os.path.exists(path):
                continue
            with open(path) as f:
                tj = json.load(f)
            if tj.get("workload") == a.workload and tj.get("spp") == spp and tj.get("pt_mode") == a.pt_mode and tj.get("kernel") == roofline_kernel:
                traffic = tj["dram_bytes_per_launch"]
                break
    except Exception:
        pass
    gtaps = taps / (kernel_ms * 1e-3) / 1e9
    roofline = {
        "bound": "hbm", "kernel": roofline_kernel,
        "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
        "traffic": traffic, "peak_source": peak_src,
        "note": "NOMINAL: SURVEY 8(d)'s algorithmic bytes over the measured HBM copy peak.  The kernel is not DRAM-bound (traffic = measured "
                "DRAM bytes per launch, orders of magnitude below the algorithmic bytes: the taps hit L1TEX/L2); what bounds it is in `gather` "
                "(texture-unit tap rate) and `issue` (SM issue slots under divergence)",
        "bytes_algo_per_launch": int(bytes_algo), "taps_per_launch": int(taps), "tf_lookups_per_launch": int(cnt["tf_lookups"]),
        "kernel_ms": round(kernel_ms, 4), "gtaps_per_s": round(gtaps, 3),
        "kernel_share_of_step": round(kernel_ms / (ms / a.steps), 4),
        "gather": dict(gather, achieved_gtaps_per_s=round(gtaps, 3), frac_of_coherent=round(gtaps / gather["coherent_gtaps_per_s"], 4),
                       frac_of_random=round(gtaps / gather["random_gtaps_per_s"], 4)),
        "issue": issue_counters(a.workload, spp, roofline_kernel),
    }

    # ---- CPU baseline: the oracle port on a bounded sample (rank 0, N = 1 only)
    cpu_baseline = None
    if world == 1 and not a.no_cpu_baseline:
        vox = vb.cpu().numpy().view(S.VOXEL_DTYPES[cfg.fmt]).reshape(cfg.n, cfg.n, cfg.n)
        cpu_baseline = cpu_port_sample(cfg, vox, base_volume, base_camera, base_lights, a.cpu_seconds)
        del vox

    # ---- the reference's own CUDA kernels on this GPU, bounded sample (context for the 3x target)
    ref_cuda = None
    if world == 1 and not a.no_ref_cuda:
        ref_cuda = reference_cuda_sample(cfg, r, 16)

    raycast = (raycast_lines(r) if not a.no_ref_cuda and not a.no_raycast else None) if world == 1 else raycast_multi
    other = other_workload_lines(r, a) if world == 1 and not a.no_ref_cuda and a.workload == "C3" else None

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,  # BASELINE.md: the reference publishes no number
        "dtype": "f32", "data": "synthetic",
        "config": {
            "workload": f"{cfg.name}: {cfg.n}^3 {['u8', 'u16', 'f16', 'f32'][cfg.fmt]} procedural {['sphere-falloff', 'CT-like', 'cloud'][cfg.gen]} volume, "
                        f"{W}x{H} path tracing, Woodcock tracking, traceDepth {depth}, one area light"
                        f"{' + constant environment light' if cfg.env else ''}, TF-{cfg.tf}, {spp} spp per step per GPU",
            "spp_per_step_per_gpu": spp, "samples_per_step": npix * spp * world,
            "parallelism": f"spp-split x{world}, volume replicated (e2e fan-out: {(e2e or {}).get('fanout')}), NCCL sum-reduce of float4 accumulators to rank 0"
                           if world > 1 else "single GPU",
            "estimator": {0: "global majorant + XORWOW (reference twin)", 1: "global majorant + Philox", 2: "macrocell local majorants + Philox"}[a.pt_mode],
            "macrocell": cell_used,
            "l2": f"volume {vb.numel() >> 20} MiB > 126 MB L2, every step renders a NEW sample range (other taps than the step before); no flush between steps",
            "image_nonzero_fraction": round(img_nonzero, 4) if img_nonzero is not None else None,
        },
        "e2e": e2e,
        "gpu_launches": int(launches),
        "clocks": clk,
        "roofline": roofline,
        "cpu_baseline": cpu_baseline,
        "reference_cuda": ref_cuda,
        "raycast": raycast,
        "other_workloads": other,
        "strong_scaling": strong,
        "c5": c5,
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def cpu_port_sample(cfg, vox, volume, camera, lights, seconds):
    """The CPU oracle (test infrastructure) timed on an image-wide bounded sample: every 16th row, as
    many frames as fit in about `seconds`.  `vox`: host numpy voxels (z, y, x); the PODs as the entry points get them."""
    from oracle import binding as B
    from sunvolumerender_b200 import scene as S

    if not os.path.exists(B.CPU_LIB):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "cpu"], stdout=subprocess.DEVNULL)
    o = B.CpuOracle(vox, cfg.fmt, (cfg.n,) * 3, volume, S.tf_table(cfg.tf), camera, lights)
    cores = B.cpu().svr_oracle_threads()
    W, H = cfg.width, cfg.height
    step = 16
    rows = len(range(8, H, step))
    t = time.perf_counter()
    o.pathtrace(cfg.trace_depth, 0, 1, rows=(8, H), row_step=step)
    dt1 = time.perf_counter() - t
    frames = int(max(1, min(4096, seconds / max(dt1, 1e-3))))
    t = time.perf_counter()
    o.pathtrace(cfg.trace_depth, 1, frames, rows=(8, H), row_step=step)
    dt = time.perf_counter() - t
    return {
        "value": W * rows * frames / dt, "unit": UNIT, "cores": int(cores), "kind": "port",
        "sample": f"rows 8,24,..(every 16th: {rows} of {H}) x {W} px x {frames} frames of {cfg.name}, global majorant + XORWOW as the reference, {dt:.1f} s",
    }


def raycast_lines(r):
    """The metric's second half: ray-cast Mrays/s on C2 (256^3 u8, 1024x1024, front-to-back compositing
    with the 1-D transfer function and gradient shading), ours and the reference's kernel_raycasting,
    device-resident, best of 5 frames; plus the image difference between the two."""
    import torch

    from oracle import binding as B
    from sunvolumerender_b200 import _lib as L
    from sunvolumerender_b200 import scene as S
    from sunvolumerender_b200.render import setup_config

    out = []
    for label, n, W, H, tf in RAYCAST_WORKLOADS:
        cfg = S.Config("RC", n, 0, 1, W, H, tf)
        setup_config(r, cfg)
        step = S.raycast_step_size()
        r.render_raycasting(step)
        torch.cuda.synchronize()

        def best_of(fn, n=5):
            best = None
            for _ in range(n):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1)
                best = ms if best is None else min(best, ms)
            return best

        ms = best_of(lambda: r.render_raycasting(step))
        # counted work of one frame (taps = trilinear fetches: 1 per step + 6 per shaded step, raycasting.cu:33,37)
        r.set_option(L.OPT_COUNTERS, 1)
        r.reset_counters()
        r.render_raycasting(step)
        torch.cuda.synchronize()
        cnt = r.counters()
        r.set_option(L.OPT_COUNTERS, 0)
        # texture-unit ceiling on this volume: coherent, dependence-free tex3D taps (svr_microbench_taps)
        sink = torch.zeros(4, dtype=torch.float32, device="cuda")
        taps_out = C.c_uint64(0)
        tex_ms = best_of(lambda: L.check(r.lib.svr_microbench_taps(C.byref(r.volume), 0, 1 << 20, 512, C.c_void_p(sink.data_ptr()), C.byref(taps_out))), 3)
        peak = taps_out.value / (tex_ms * 1e-3) / 1e9
        line = {"workload": label, "value": cfg.width * cfg.height / (ms * 1e-3) / 1e6,
                "unit": "Mrays/s", "ms_per_frame": ms, "steps": cnt["steps"], "steps_skipped_as_empty": cnt["skipped"],
                "taps": cnt["shade_taps"], "tf_lookups": cnt["tf_lookups"],
                "roofline": {"bound": "l1tex", "achieved": cnt["shade_taps"] / (ms * 1e-3) / 1e9, "peak": peak, "unit": "Gtaps/s",
                             "frac": cnt["shade_taps"] / (ms * 1e-3) / 1e9 / peak,
                             "peak_source": "measured here: 2^20 threads x 512 coherent tex3D taps on the same volume"}}
        try:
            ref = B.RefCuda(cfg.width, cfg.height)
            ref.setup(r.volume, r.tf, r.camera, r.lights, r.env)
            ref.render_raycasting(step)
            torch.cuda.synchronize()
            rms = best_of(lambda: ref.render_raycasting(step))
            line["reference_cuda"] = {"value": cfg.width * cfg.height / (rms * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_frame": rms}
            line["max_u8_diff_vs_reference"] = int((r.ldr_image().int() - ref.ldr_image().int()).abs().max())
        except (FileNotFoundError, OSError) as e:
            line["reference_cuda"] = {"unavailable": str(e)}
        out.append(line)
    return out


def _best_ms(fn, reps=3, warm=1):
    import torch

    best = None
    for i in range(reps + warm):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn(i)
        e1.record()
        torch.cuda.synchronize()
        if i >= warm:
            ms = e0.elapsed_time(e1)
            best = ms if best is None else min(best, ms)
    return best


def other_workload_lines(r, a):
    """The driver-run record of what the headline does not show (one GPU, device-resident, the reference's kernels beside
    every line on the same scene):
      * C3 with the camera moved in so that the body fills the frame (no sky to classify away);
      * the drop-in protocol: the workload as a reference host renders it, one render_pathtracer call per sample;
      * C4 (configs[3]) at its full 512 spp, with counted taps and its roofline;
      * C1 (configs[0]): ray cast + 16-spp path trace;
      * the reference built with its shipped -maxrregcount=32 beside the uncapped build."""
    import torch

    from sunvolumerender_b200 import _lib as L
    from sunvolumerender_b200 import scene as S
    from sunvolumerender_b200.render import setup_config

    out = []
    peak, _ = measured_peak()

    def counted(cfg, spp, first=0):
        r.set_option(L.OPT_COUNTERS, 1)
        r.reset_counters()
        buf = torch.zeros(cfg.width * cfg.height * 4, dtype=torch.float32, device="cuda")
        r.accumulate(buf, cfg.trace_depth, first, spp, clear=True)
        torch.cuda.synchronize()
        c = r.counters()
        r.set_option(L.OPT_COUNTERS, 0)
        return c

    # ---- C3, close view and drop-in protocol
    cfg = S.CONFIGS["C3"]
    vb3 = setup_config(r, cfg)
    layouts = {"workload": "voxel layout study: independent trilinear taps on the benched volumes, three storages (see layout_study)",
               "C3_512^3_u16": layout_study(r, vb3, cfg.n)}
    del vb3
    npix = cfg.width * cfg.height
    buf = torch.zeros(npix * 4, dtype=torch.float32, device="cuda")
    cam0 = r.camera
    r.set_camera(S.make_camera((0, 0, cam0.pos.z * 0.45), (1, 0, 0), (0, 1, 0), (0, 0, 1), 45.0, 0.0, 1.0, 1.0, cfg.width, cfg.height))
    ms = _best_ms(lambda i: r.accumulate(buf, cfg.trace_depth, i * cfg.spp, cfg.spp, clear=True))
    c = counted(cfg, cfg.spp)
    bytes_algo, taps = algorithmic_bytes(c, cfg.voxel_bytes, npix)
    out.append({"workload": f"C3 close view: camera at 0.45 x the framing distance, the body fills the frame ({c['scatters'] / c['paths']:.2f} scatter events per "
                            f"sample against {0.104:.2f} in the default view), {cfg.spp} spp per launch, device-resident",
                "value": npix * cfg.spp / (ms * 1e-3), "unit": UNIT, "ms_per_launch": ms,
                "roofline": {"bound": "hbm", "achieved": bytes_algo / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": bytes_algo / (ms * 1e-3) / 1e9 / peak,
                             "taps_per_launch": int(taps), "gtaps_per_s": taps / (ms * 1e-3) / 1e9, "note": "nominal, see the headline's roofline.note"},
                "reference_cuda": reference_cuda_sample(cfg, r, 16)})
    r.set_camera(cam0)

    def protocol(i):
        r.frame_no = 0
        for _ in range(cfg.spp):
            r.render_pathtracer(cfg.trace_depth)   # Canvas::paintGL: one call = one sample, running mean + tone map every call

    l0, b0 = r.launch_count(), r.lib.svr_lookahead_batch_count()
    ms = _best_ms(protocol, reps=2)
    per_step = (r.launch_count() - l0) // 3, (r.lib.svr_lookahead_batch_count() - b0) // 3   # _best_ms: one warm-up + reps passes
    r.set_option(L.OPT_PT_LOOKAHEAD, 0)
    ms_plain = _best_ms(protocol, reps=2)
    r.set_option(L.OPT_PT_LOOKAHEAD, 32)
    out.append({"workload": f"C3 through the drop-in protocol: {cfg.spp} x render_pathtracer(img, renderParams), 1 spp per call, running mean and tone-mapped image "
                            f"after every call, one final sync.  Library defaults: the lane-per-pixel kernel for the first 16 calls, then 32 samples ahead per "
                            f"sample-parallel launch and one fold per call (SVR_OPT_PT_LOOKAHEAD; hdrBuffer and image bit-identical to one sample per call)",
                "value": npix * cfg.spp / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "launches_per_step": per_step[0], "lookahead_batches_per_step": per_step[1],
                "ms_per_step_one_sample_per_launch": ms_plain,
                "reference_cuda": reference_cuda_sample(cfg, r, cfg.spp, reps=2)})
    ref_r32 = reference_cuda_sample(cfg, r, 16, r32=True)
    out.append({"workload": "C3, variants of the reference's kernels beside the unmodified uncapped build the headline ratio uses: built with the shipped "
                            "-maxrregcount=32 (CMakeLists.txt:9); and the environment twin, which renders the very lighting this arm renders (area + environment)",
                "reference_cuda_r32": ref_r32, "reference_cuda_env_twin": reference_cuda_sample(cfg, r, 16, env=True), "reference_cuda": reference_cuda_sample(cfg, r, 16)})
    del buf

    # ---- C4 at its full 512 spp: 4 launches of 128
    cfg = S.CONFIGS["C4"]
    try:
        vb4 = setup_config(r, cfg)
        layouts["C4_1024^3_f16_bits"] = layout_study(r, vb4, cfg.n)
        del vb4
        torch.cuda.empty_cache()
        npix = cfg.width * cfg.height
        per, launches = cfg.spp, 1   # one launch renders the config's 512 spp (4 launches of 128: 12 % slower, the per-pixel drains repeat)
        buf = torch.zeros(npix * 4, dtype=torch.float32, device="cuda")

        def c4_step(i):
            for j in range(launches):
                r.accumulate(buf, cfg.trace_depth, (i * launches + j) * per, per, clear=(j == 0))

        ms = _best_ms(c4_step, reps=2)
        c = counted(cfg, per)
        bytes_algo, taps = algorithmic_bytes(c, cfg.voxel_bytes, npix)
        bytes_algo, taps = bytes_algo * launches, taps * launches
        gather = gather_ceilings(r)
        g = taps / (ms * 1e-3) / 1e9
        out.append({"workload": f"C4: 1024^3 f16 cloud, 1920x1080, traceDepth {cfg.trace_depth}, {cfg.spp} spp per step in {launches} launch{'es' if launches > 1 else ''}, "
                                f"device-resident, scatter-queue kernel",
                    "value": npix * cfg.spp / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "macrocell": grid_cell(r),
                    "counted": {"taps_per_step": int(taps), "scatter_events_per_sample": c["scatters"] / c["paths"], "cell_visits_per_sample": c["cells"] / c["paths"]},
                    "roofline": {"bound": "hbm", "achieved": bytes_algo / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": bytes_algo / (ms * 1e-3) / 1e9 / peak,
                                 "gtaps_per_s": g, "gather": dict(gather, frac_of_coherent=g / gather["coherent_gtaps_per_s"], frac_of_random=g / gather["random_gtaps_per_s"]),
                                 "issue": issue_counters("C4", 128, "pathtrace_queue_kernel<0>"), "note": "nominal; taps counted on a launch of the same size"},
                    "reference_cuda": reference_cuda_sample(cfg, r, 8)})
        del buf
    except Exception as e:  # e.g. not enough device memory beside the other buffers
        out.append({"workload": "C4", "unavailable": str(e)})

    # ---- C1: ray cast + 16-spp path trace
    cfg = S.CONFIGS["C1"]
    setup_config(r, cfg)
    torch.cuda.empty_cache()
    npix = cfg.width * cfg.height
    buf = torch.zeros(npix * 4, dtype=torch.float32, device="cuda")
    step = S.raycast_step_size()
    ms_rc = _best_ms(lambda i: r.render_raycasting(step), reps=5)
    r.set_option(L.OPT_PT_WARP_MIN_SPP, 16)
    ms_pt = _best_ms(lambda i: r.accumulate(buf, cfg.trace_depth, i * cfg.spp, cfg.spp, clear=True), reps=5)
    r.set_option(L.OPT_PT_WARP_MIN_SPP, 32)
    ms_pt_mega = _best_ms(lambda i: r.accumulate(buf, cfg.trace_depth, i * cfg.spp, cfg.spp, clear=True), reps=5)
    line = {"workload": f"C1: 128^3 u8 sphere, 512x512, one area light: front-to-back ray cast, and a {cfg.spp}-spp path trace in one launch",
            "raycast": {"value": npix / (ms_rc * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_frame": ms_rc},
            "pathtrace": {"value": npix * cfg.spp / (min(ms_pt, ms_pt_mega) * 1e-3), "unit": UNIT, "ms_per_launch": min(ms_pt, ms_pt_mega),
                          "ms_sample_parallel_kernel": ms_pt, "ms_lane_per_pixel_kernel": ms_pt_mega},
            "reference_cuda": reference_cuda_sample(cfg, r, cfg.spp)}
    try:
        from oracle import binding as B

        ref = B.RefCuda(cfg.width, cfg.height)
        ref.setup(r.volume, r.tf, r.camera, r.lights, r.env)
        ms_ref = _best_ms(lambda i: ref.render_raycasting(step), reps=5)
        line["reference_cuda_raycast"] = {"value": npix / (ms_ref * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_frame": ms_ref}
    except (FileNotFoundError, OSError) as e:
        line["reference_cuda_raycast"] = {"unavailable": str(e)}
    out.append(line)
    out.append(layouts)
    return out


RAYCAST_WORKLOADS = [
    # (label, volume edge, width, height, transfer function)
    ("C2: 256^3 u8 CT-like volume, 1024x1024, TF-thin", 256, 1024, 1024, "thin"),
    ("C2: 256^3 u8 CT-like volume, 1024x1024, TF-default", 256, 1024, 1024, "default"),
    ("RC4K: 512^3 u8 CT-like volume, 3840x2160, TF-thin (a frame long enough for a split to pay)", 512, 3840, 2160, "thin"),
]


def raycast_lines_multi(r, rank, world, dev):
    """Ray casting on N GPUs (the metric's "ray-cast Mrays/s at 1/2/4/8 B200"): the volume replicated, the image split
    across the ranks (one deterministic pass, SURVEY.md section 8e), three ways of putting it together on rank 0:
      gather   contiguous row blocks, NCCL gather of the u8 blocks;
      reduce   row bands dealt out round robin (balanced), NCCL sum-reduce of the u8 images (disjoint bands: a gather);
      peer     the same bands written STRAIGHT into rank 0's image through peer mappings over NVLink, completion by a flag in
               rank 0's memory (distributed.PeerFrame): no collective, no host in the loop.
    Timed per frame with CUDA events, max over ranks, best of 10 frames; rank 0 also renders the whole frame alone and
    every assembled image must equal it bit for bit."""
    import torch
    import torch.distributed as dist

    from sunvolumerender_b200 import _lib as L
    from sunvolumerender_b200 import distributed as D
    from sunvolumerender_b200 import scene as S
    from sunvolumerender_b200.render import setup_config

    def best_frame(frame, n=10):
        frame()
        torch.cuda.synchronize()
        best = None
        for _ in range(n):
            dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            frame()
            e1.record()
            torch.cuda.synchronize()
            ms = D.max_over_ranks(e0.elapsed_time(e1), dev)
            best = ms if best is None else min(best, ms)
        return best

    out = []
    for label, n, W, H, tf in RAYCAST_WORKLOADS:
        cfg = S.Config("RC", n, L.VOXEL_U8, L.GEN_CT, W, H, tf)
        setup_config(r, cfg)
        step = S.raycast_step_size()
        rows = S.split_rows(H, world)
        y0, y1 = rows[rank]
        pad = max(b - a for a, b in rows)
        block = torch.zeros(pad * W * 4, dtype=torch.uint8, device=dev)
        gathered = [torch.zeros_like(block) for _ in range(world)] if rank == 0 else None
        img = r.img.view(H, W, 4)
        even = all(b - a == pad for a, b in rows)
        mine = r.img[y0 * W * 4: y1 * W * 4] if even else block   # a rank's rows are contiguous in the image
        r.render_raycasting(step)   # builds the macrocell grid; the single-GPU image
        torch.cuda.synchronize()
        single = r.ldr_image().clone() if rank == 0 else None

        def frame_gather():
            r.render_raycasting_f32(None, step, rows=(y0, y1), img=r.img)   # this rank's rows of the u8 image
            if not even:
                block[: (y1 - y0) * W * 4].copy_(img[y0:y1].reshape(-1))
            dist.gather(mine, gathered, dst=0)

        ms_gather = best_frame(frame_gather)
        eq_gather = bool(torch.equal(torch.cat([g[: (b - a) * W * 4] for g, (a, b) in zip(gathered, rows)]).view(H, W, 4), single)) if rank == 0 else None

        def frame_reduce():
            r.img.zero_()
            r.render_raycasting_bands(rank, world, step)
            dist.reduce(r.img, dst=0, op=dist.ReduceOp.SUM)

        ms_reduce = best_frame(frame_reduce)
        eq_reduce = bool(torch.equal(r.ldr_image(), single)) if rank == 0 else None

        ms_peer, eq_peer, peer_err = None, None, None
        try:
            pf = D.PeerFrame(r, W * H * 4)

            def frame_peer():
                r.render_raycasting_bands(rank, world, step, img_ptr=pf.img_ptr)
                pf.frame_done()

            ms_peer = best_frame(frame_peer)
            if rank == 0:
                eq_peer = bool(torch.equal(pf.image().view(H, W, 4), single))
            pf.close()
        except Exception as e:  # no peer access between these GPUs
            peer_err = str(e)
        times = {"gather": ms_gather, "reduce": ms_reduce}
        if ms_peer is not None:
            times["peer"] = ms_peer
        how = min(times, key=times.get)
        out.append({"workload": f"{label}, x{world} GPUs", "value": W * H / (times[how] * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_frame": times[how], "assembled_by": how,
                    "ms_per_frame_contiguous_rows_nccl_gather": ms_gather, "ms_per_frame_interleaved_bands_nccl_reduce": ms_reduce,
                    "ms_per_frame_interleaved_bands_peer_writes": ms_peer, "peer_unavailable": peer_err,
                    "equals_single_gpu_image": bool(eq_gather and eq_reduce and (eq_peer is not False)) if rank == 0 else None})
    return out


def reference_cuda_sample(cfg, r, frames, reps=3, r32=False, env=False):
    import torch

    from oracle import binding as B

    try:
        ref = B.RefCuda(cfg.width, cfg.height, r32=r32, env=env)
    except (FileNotFoundError, OSError) as e:
        return {"unavailable": str(e)}
    ref.setup(r.volume, r.tf, r.camera, r.lights, r.env)
    ref.render_pathtracer(2, cfg.trace_depth)
    torch.cuda.synchronize()
    best = None
    for _ in range(reps):
        ref.frame_no = 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ref.render_pathtracer(frames, cfg.trace_depth)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        best = ms if best is None else min(best, ms)
    return {"value": cfg.width * cfg.height * frames / (best * 1e-3), "unit": UNIT, "ms": best,
            "sample": f"{frames} frames (render_pathtracer x{frames}, 3 launches each) of {cfg.name}{', -maxrregcount=32' if r32 else ''}, "
                      + ("ENVIRONMENT TWIN: the reference's sources with the line commented out at pathtracer.cu:233 re-enabled (oracle/Makefile), i.e. the same "
                         "area + environment lighting this arm renders" if env else "env light off (dead code in the reference)") + f", best of {reps}"}


# ------------------------------------------------------------------------------------------------
# reference arm
# ------------------------------------------------------------------------------------------------
def run_reference(a):
    rank = env_int("RANK", 0)
    if rank != 0:
        return  # the reference is single-device: rank 0 alone runs it
    import numpy as np
    import torch

    from oracle import binding as B                 # the checkers: the reference's kernels + the plain-cudart scene builder
    from sunvolumerender_b200 import scene as S     # host-side scene description only (numpy / ctypes structs); the product
    #                                                 library libsvr_b200.so is NOT loaded anywhere in this arm

    cfg = S.CONFIGS[a.workload]
    spp = a.spp or cfg.spp
    W, H = cfg.width, cfg.height
    base = {"impl": "reference", "metric": METRIC, "unit": UNIT, "n_gpus": 1, "steps": a.steps, "warmup": a.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic"}
    if not torch.cuda.is_available():
        emit({"impl": "reference", "unavailable": "no CUDA device: the reference's only implementation of the path is CUDA"})
        return
    local = env_int("LOCAL_RANK", 0)
    torch.cuda.set_device(local)
    torch.zeros(1, device="cuda")  # the primary context the runtime-API calls below share
    try:
        scene = B.RefScene(cfg, S.tf_table(cfg.tf))  # cudaArray + texture objects with the reference loaders' descriptors, synthetic voxels
    except (FileNotFoundError, OSError) as e:
        emit({"impl": "reference", "unavailable": f"oracle/_ref/libsvr_refscene.so not prebuilt: {e}"})
        return
    camera = S.default_camera(cfg.extent, W, H)
    lights = [S.default_area_light(cfg.extent)]
    env = S.constant_env_light()
    if a.ref_device == "cpu":
        vox = scene.download(S.VOXEL_DTYPES[cfg.fmt], cfg.n)
        cb = cpu_port_sample(cfg, vox, scene.volume, camera, lights, max(10.0, a.cpu_seconds))
        line = dict(base, value=cb["value"], ms_per_step=None,
                    config={"workload": f"{cfg.name} (bounded sample: {cb['sample']})"},
                    cpu_baseline=cb, e2e={"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
        emit(line)
        return
    try:
        ref = B.RefCuda(W, H, r32=a.ref_r32)
    except (FileNotFoundError, OSError) as e:
        emit({"impl": "reference", "unavailable": f"oracle/_ref library for {W}x{H} not prebuilt: {e}"})
        return
    ref.setup(scene.volume, scene.tf, camera, lights, env)
    clocks = ClockSampler(local)

    def step():
        ref.frame_no = 0
        ref.render_pathtracer(spp, cfg.trace_depth)  # Canvas::paintGL's loop: one render_pathtracer per sample

    for _ in range(a.warmup):
        step()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    ev0.record()
    for _ in range(a.steps):
        step()
    ev1.record()
    torch.cuda.synchronize()
    t1 = time.time()
    clocks.window(t0, t1)
    ms = ev0.elapsed_time(ev1)
    HB = ref.HB
    value = W * H * spp * a.steps / (ms * 1e-3)
    nz = float((ref.ldr_image()[..., :3] > 0).float().mean())
    line = dict(
        base, value=value, ms_per_step=ms / a.steps,
        config={"workload": f"{cfg.name}: {cfg.n}^3 {['u8', 'u16', 'f16', 'f32'][cfg.fmt]}, {W}x{H} path tracing, traceDepth {cfg.trace_depth}, one area light (environment light is dead "
                            f"code in the reference, pathtracer.cu:233), {spp} spp per step; the reference's unmodified kernels, sm_100, "
                            f"-use_fast_math{' -maxrregcount=32' if a.ref_r32 else ''}; canvas {W}x{HB} (no bounds guard), {W}x{H} counted; scene built by "
                            f"oracle/ref_scene.cu (plain CUDA runtime, same voxels as the other arm's generator)",
                "spp_per_step_per_gpu": spp, "samples_per_step": W * H * spp, "image_nonzero_fraction": round(nz, 4)},
        e2e={"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        gpu_launches=3 * spp * a.steps,
        clocks=clocks.finish(),
        cpu_baseline={"value": value, "unit": UNIT, "cores": 0, "kind": "reference",
                      "sample": "the reference has no CPU path; this is its own CUDA implementation (oracle/_ref) on one B200, full workload"},
    )
    emit(line)
    scene.close()
    if os.environ.get("SVR_BENCH_PRINT_MAPS"):  # which of this repository's libraries the arm's process mapped
        with open("/proc/self/maps") as f:
            libs = sorted({ln.split()[-1] for ln in f if "svr" in ln and ".so" in ln})
        print("mapped:", libs, file=sys.stderr)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, images):
    """Writes each (H, W, C) image as out_dir/<name>.npy in float32.  Above DUMP_LIMIT_BYTES in all, the same fixed,
    seeded sample of pixels is written for every image, with its flat pixel indices as pixel_index.npy (float64), so that
    two builds run with the same arguments can be compared output for output."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    arrays = {name: img.float().cpu().numpy() for name, img in images.items()}
    total = sum(v.size * 4 for v in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        H, W = next(iter(arrays.values())).shape[:2]
        keep = int(H * W * (DUMP_LIMIT_BYTES - 4096) // (total + 8 * H * W))  # 4 KiB for the .npy headers
        idx = np.sort(np.random.default_rng(0).choice(H * W, size=keep, replace=False))
        arrays = {name: v.reshape(H * W, -1)[idx] for name, v in arrays.items()}
        arrays["pixel_index"] = idx.astype(np.float64)
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), v)


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line of the contract, on the process's real stdout."""
    text = json.dumps(line) + "\n"
    if _REAL_STDOUT is None:
        sys.stdout.write(text)
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, text.encode())


def main():
    # Libraries write to stdout behind Python's back (NCCL's "NCCL version ..." banner at communicator creation): route
    # file descriptor 1 to stderr for the whole run and keep the real stdout for the one JSON line.
    global _REAL_STDOUT
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C3")
    ap.add_argument("--spp", type=int, default=0, help="samples per pixel per step per GPU (0 = the workload's)")
    ap.add_argument("--pt-mode", type=int, default=2, choices=[0, 1, 2])
    ap.add_argument("--cell", type=int, default=0, help="macrocell edge in voxels (0 = the library default)")
    ap.add_argument("--e2e-fanout", default="p2p", choices=["p2p", "nvlink", "pcie"],
                    help="N > 1, e2e: how the voxels reach every GPU: one PCIe upload + copy-engine pushes over NVLink (p2p), "
                         "one PCIe upload + NCCL broadcast (nvlink), or one PCIe upload per rank (pcie)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--force-e2e", action="store_true", help="run the e2e leg for volumes above 2 GiB too (pins that much host memory per rank)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-cuda", action="store_true")
    ap.add_argument("--no-raycast", action="store_true")
    ap.add_argument("--no-c5", action="store_true", help="N = 8: skip the C5 line (2048^3 u16, 4K, 1024 spp over the GPUs)")
    ap.add_argument("--c5", action="store_true", help="run the C5 line at any N > 1")
    ap.add_argument("--ref-device", default="cuda", choices=["cuda", "cpu"])
    ap.add_argument("--ref-r32", action="store_true", help="reference built with the shipped -maxrregcount=32")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the HDR and tone-mapped images of the last timed step as DIR/<name>.npy (float32)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the product's timed path (--impl ours)")
    a.warmup = max(a.warmup, 0)
    world = env_int("WORLD_SIZE", 1)
    if a.impl == "ours" and world != a.gpus and world == 1 and a.gpus > 1:
        # launched without torchrun: re-launch ourselves the way the driver would
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={a.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", str(29500 + os.getpid() % 1000), os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
