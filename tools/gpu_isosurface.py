"""Isosurface (svr_render_isosurface) on C2 (256^3 u8 CT, 1024 x 1024) and C3 (512^3 u16 CT, 1920 x 1080), each in the default
view and the close view (camera at 0.45 x the framing distance, as tools/gpu_projection.py).

Per threshold (0.15: skin, 0.7: bone) with skipping on and off (SVR_OPT_RC_SKIP):
  * ms per frame: CUDA events around 10 frames, best of 5 windows after a warm-up;
  * M rays/s over that time;
  * from a separate counters run (SVR_OPT_COUNTERS): the share of steps skipped, taken samples per ray;
  * the share of rays that hit;
  * render_raycasting of the configuration's transfer function on the same frame, for comparison.
Checks that image and surface are bit-identical with skipping on and off.  Prints the card and its power limit, then a markdown
table; --json PATH also writes the results."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sunvolumerender_b200 import _lib as L  # noqa: E402
from sunvolumerender_b200 import scene as S  # noqa: E402
from sunvolumerender_b200.render import Renderer, setup_config  # noqa: E402

THRESHOLDS = (0.15, 0.7)


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
        step = S.raycast_step_size(r.volume.spacing.tuple())
        surface = torch.empty(cfg.width * cfg.height * 4, dtype=torch.float32, device="cuda")
        base = S.default_camera(cfg.extent, cfg.width, cfg.height)
        for view in ("default", "close"):
            cam = base if view == "default" else S.make_camera((0.0, 0.0, 0.45 * base.pos.z), (1, 0, 0), (0, 1, 0), (0, 0, 1), 45.0, 0.0, 1.0, 1.0,
                                                               cfg.width, cfg.height)
            r.set_camera(cam)
            r.set_option(L.OPT_RC_SKIP, 1)
            rc_ms = events(lambda: r.render_raycasting(step))
            for iso in THRESHOLDS:
                outputs = {}
                for skip in (1, 0):
                    r.set_option(L.OPT_RC_SKIP, skip)
                    fn = lambda: r.render_isosurface(iso, step, surface=surface)  # noqa: E731
                    ms = events(fn)
                    c = counted(r, fn)
                    outputs[skip] = (surface.clone(), r.img.clone())
                    hits = int(torch.isfinite(surface.view(-1, 4)[:, 3]).sum())
                    row = {"config": cname, "view": view, "iso": iso, "skip": skip, "ms": round(ms, 4),
                           "mrays_per_s": round(c["paths"] / (ms * 1e-3) / 1e6, 1), "skipped_share": round(c["skipped"] / max(c["steps"], 1), 4),
                           "taps_per_ray": round(c["shade_taps"] / max(c["paths"], 1), 1), "hit_share": round(hits / max(c["paths"], 1), 4),
                           "cells": c["cells"], "raycast_ms": round(rc_ms, 4)}
                    rows.append(row)
                    print(json.dumps(row), flush=True)
                assert torch.equal(outputs[0][0], outputs[1][0]) and torch.equal(outputs[0][1], outputs[1][1]), (cname, view, iso)
    r.set_option(L.OPT_RC_SKIP, 1)
    results["rows"] = rows
    print()
    print(f"{name}, {power}")
    print("| config | view | iso | skip | ms | M rays/s | steps skipped | taps per ray | hits | render_raycasting ms |")
    print("|---|---|---|---|---|---|---|---|---|---|")
    for x in rows:
        print(f"| {x['config']} | {x['view']} | {x['iso']} | {'on' if x['skip'] else 'off'} | {x['ms']:.3f} | {x['mrays_per_s']:.0f} | "
              f"{x['skipped_share']:.3f} | {x['taps_per_ray']:.1f} | {x['hit_share']:.3f} | {x['raycast_ms']:.3f} |")
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(results, f, indent=1)
    r.close()


if __name__ == "__main__":
    main()
