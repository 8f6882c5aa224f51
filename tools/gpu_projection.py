"""Intensity projections (svr_render_projection) on C2 (256^3 u8 CT, 1024 x 1024) and C3 (512^3 u16 CT, 1920 x 1080), each in
the default view and the close view (camera at 0.45 x the framing distance, as tools/gpu_progressive_denoise.py).

Per mode (max, min, mean) with skipping on and off (SVR_OPT_RC_SKIP):
  * ms per frame: CUDA events around 10 frames, best of 5 windows after a warm-up;
  * M rays/s and G taps/s: rays and executed taps from a separate counters run (SVR_OPT_COUNTERS), over the timed frame;
  * the share of steps skipped;
  * taps/s as a share of the coherent tex3D ceiling on the same volume (svr_microbench_taps, 2^20 threads x 512 taps, best
    of 3);
  * render_raycasting of the configuration's transfer function on the same frame, for comparison.
Prints the card and its power limit, then a markdown table; --json PATH also writes the results."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sunvolumerender_b200 import _lib as L  # noqa: E402
from sunvolumerender_b200 import scene as S  # noqa: E402
from sunvolumerender_b200.render import Renderer, setup_config  # noqa: E402

MODES = ("max", "min", "mean")


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return name, q.stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers below still stand; the power limit is then unknown
        return name, f"power limit unavailable ({e})"


def events(fn, frames=10, windows=5):
    fn()
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(windows):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(frames):
            fn()
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1) / frames)
    return best


def counted(r, fn):
    r.set_option(L.OPT_COUNTERS, 1)
    r.reset_counters()
    fn()
    torch.cuda.synchronize()
    c = r.counters()
    r.set_option(L.OPT_COUNTERS, 0)
    return c


def coherent_ceiling(r):
    sink = torch.zeros(1 << 20, dtype=torch.float32, device="cuda")
    taps = C.c_uint64(0)

    def run():
        L.check(r.lib.svr_microbench_taps(C.byref(r.volume), 0, 1 << 20, 512, C.c_void_p(sink.data_ptr()), C.byref(taps)), "svr_microbench_taps")

    ms = events(run, frames=1, windows=3)
    return taps.value / (ms * 1e-3) / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    name, power = card()
    print(f"card: {name}; power.limit, clocks.max.sm: {power}", flush=True)
    r = Renderer(0)
    results = {"card": name, "power": power, "rows": []}
    rows = []
    for cname in ("C2", "C3"):
        cfg = S.CONFIGS[cname]
        setup_config(r, cfg)
        r.set_option(L.OPT_MACROCELL_SIZE, 0)
        ceiling = coherent_ceiling(r)
        step = S.raycast_step_size(r.volume.spacing.tuple())
        out = torch.empty(cfg.width * cfg.height, dtype=torch.float32, device="cuda")
        base = S.default_camera(cfg.extent, cfg.width, cfg.height)
        for view in ("default", "close"):
            cam = base if view == "default" else S.make_camera((0.0, 0.0, 0.45 * base.pos.z), (1, 0, 0), (0, 1, 0), (0, 0, 1), 45.0, 0.0, 1.0, 1.0,
                                                               cfg.width, cfg.height)
            r.set_camera(cam)
            r.set_option(L.OPT_RC_SKIP, 1)
            rc_ms = events(lambda: r.render_raycasting(step))
            for mode in MODES:
                values = {}
                for skip in (1, 0):
                    r.set_option(L.OPT_RC_SKIP, skip)
                    fn = lambda: r.render_projection(mode, (0.5, 1.0), step, out=out)  # noqa: E731
                    ms = events(fn)
                    c = counted(r, fn)
                    values[skip] = out.clone()
                    gtaps = c["shade_taps"] / (ms * 1e-3) / 1e9
                    row = {"config": cname, "view": view, "mode": mode, "skip": skip, "ms": round(ms, 4),
                           "mrays_per_s": round(c["paths"] / (ms * 1e-3) / 1e6, 1), "gtaps_per_s": round(gtaps, 2),
                           "skipped_share": round(c["skipped"] / max(c["steps"], 1), 4), "cells": c["cells"],
                           "share_of_coherent_ceiling": round(gtaps / ceiling, 3), "coherent_ceiling_gtaps_per_s": round(ceiling, 1),
                           "raycast_ms": round(rc_ms, 4)}
                    rows.append(row)
                    print(json.dumps(row), flush=True)
                assert torch.equal(values[0], values[1]), (cname, view, mode)
    r.set_option(L.OPT_RC_SKIP, 1)
    results["rows"] = rows
    print()
    print(f"{name}, {power}")
    print("| config | view | mode | skip | ms | M rays/s | G taps/s | steps skipped | share of coherent ceiling | render_raycasting ms |")
    print("|---|---|---|---|---|---|---|---|---|---|")
    for x in rows:
        print(f"| {x['config']} | {x['view']} | {x['mode']} | {'on' if x['skip'] else 'off'} | {x['ms']:.3f} | {x['mrays_per_s']:.0f} | "
              f"{x['gtaps_per_s']:.1f} | {x['skipped_share']:.3f} | {x['share_of_coherent_ceiling']:.2f} | {x['raycast_ms']:.3f} |")
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(results, f, indent=1)
    r.close()


if __name__ == "__main__":
    main()
