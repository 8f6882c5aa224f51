"""Curved planar reformation (svr_render_curved) on C3 (512^3 u16 CT, 256 MB of voxels: more than the 126 MB L2), along a smooth
curve through the body (2000 points, 581 voxels long):
  * a thin straightened 1024 x 512 CPR (half a voxel per pixel across, one row per station), and svr_render_slices of a thin
    1024 x 512 axial slice at the same spacing: the same pixel count, one fetch per pixel;
  * 16- and 64-sample MIP and AIP slabs of that CPR (one sample per voxel), with skipping (SVR_OPT_RC_SKIP) on and off, alone and
    as 16-angle stacks (one call: the per-call host work of computing and staging the frames is then small beside the kernel);
    value and image are checked equal with torch.equal;
  * a 36-angle rotational stack of thin 512 x 512 straightened images (10 degrees apart);
  * 256 thin cross-sections of 128 x 128 (half a voxel per pixel);
  * the host time of svr_curve_frames for 16384 stations (no GPU work).
Per row: ms per call (CUDA events around 10 calls, best of 5 windows after a warm-up), G taps/s (executed taps from a separate
counters run, over the timed call), the share of steps skipped, and taps/s as a share of the coherent tex3D ceiling on the same
volume (svr_microbench_taps, as tools/gpu_projection.py).  Prints the card and its power limit, then a markdown table; --json PATH
also writes the results."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sunvolumerender_b200 import _lib as L  # noqa: E402
from sunvolumerender_b200 import scene as S  # noqa: E402
from sunvolumerender_b200.render import Renderer, setup_config  # noqa: E402

from gpu_projection import card, coherent_ceiling, counted, events  # noqa: E402


def body_curve(n, m=2000):
    u = np.linspace(0.0, 1.0, m)
    return np.stack([0.18 * n * np.sin(2 * np.pi * u), (u - 0.5) * 0.8 * n, 0.1 * n * np.cos(np.pi * u)], 1).astype(np.float32)


def cases(n, pts):
    L_ = S.polyline_length(pts)

    def cpr(slab=0, mode="max", w=1024, h=512, count=1):
        return S.straightened_curve(w, h, 0.5, station_spacing=L_ / h, up=(0, 0, 1), count=count, angle_step=np.pi / 18,
                                    thickness=float(slab), sample_spacing=1.0, mode=mode)

    out = [("thin CPR 1024 x 512", "curved", cpr())]
    axial = S.axis_slice((n, n, n), (1, 1, 1), "z", n // 2)
    axial.imageW, axial.imageH = 1024, 512
    axial.axisU[0] = axial.axisV[1] = 0.5
    out.append(("thin slice 1024 x 512", "slices", axial))
    for slab in (16, 64):
        for mode in ("max", "mean"):
            out.append((f"CPR slab {slab} {'MIP' if mode == 'max' else 'AIP'}", "curved", cpr(slab, mode)))
    for slab in (16, 64):  # 16 angles per call: the kernel, not the per-call host work, sets the time
        for mode in ("max", "mean"):
            out.append((f"CPR slab {slab} {'MIP' if mode == 'max' else 'AIP'} x 16 angles", "curved", cpr(slab, mode, count=16)))
    out.append(("rotational 36 x 512^2", "curved", cpr(w=512, h=512, count=36)))
    out.append(("cross 256 x 128^2", "curved", S.curve_cross_sections(128, 128, 256, 0.5, L_ / 256, up=(0, 0, 1))))
    return out


def frames_host_ms(pts, stations=16384, reps=20):
    L_ = S.polyline_length(pts)
    S.curve_frames(pts, (0, 0, 1), L_ / stations, stations)
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        S.curve_frames(pts, (0, 0, 1), L_ / stations, stations)
        best = min(best, (time.perf_counter() - t0) * 1e3)
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    name, power = card()
    print(f"card: {name}; power.limit, clocks.max.sm: {power}", flush=True)
    r = Renderer(0)
    cfg = S.CONFIGS["C3"]
    setup_config(r, cfg)
    r.set_option(L.OPT_MACROCELL_SIZE, 0)
    ceiling = coherent_ceiling(r)
    pts = body_curve(cfg.n)
    print(f"curve length {S.polyline_length(pts):.1f}", flush=True)
    rows = []
    for what, kind, p in cases(cfg.n, pts):
        shape = (p.count, p.imageH, p.imageW)
        value = torch.empty(shape, dtype=torch.float32, device="cuda")
        img = torch.empty(shape + (4,), dtype=torch.uint8, device="cuda")
        outs = {}
        for skip in ((1, 0) if p.thickness > 0 else (1,)):
            r.set_option(L.OPT_RC_SKIP, skip)
            if kind == "curved":
                fn = lambda: r.render_curved(pts, p, value, img)  # noqa: E731
            else:
                fn = lambda: r.render_slices(p, value, img)  # noqa: E731
            ms = events(fn)
            c = counted(r, fn)
            outs[skip] = (value.clone(), img.clone())
            gtaps = c["shade_taps"] / (ms * 1e-3) / 1e9
            row = {"case": what, "skip": skip if p.thickness > 0 else None, "ms": round(ms, 4), "pixels": c["paths"],
                   "gtaps_per_s": round(gtaps, 2), "skipped_share": round(c["skipped"] / max(c["steps"], 1), 4), "steps": c["steps"],
                   "share_of_coherent_ceiling": round(gtaps / ceiling, 3), "coherent_ceiling_gtaps_per_s": round(ceiling, 1)}
            rows.append(row)
            print(json.dumps(row), flush=True)
        if len(outs) == 2:
            assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]), what
        del value, img, outs
    r.set_option(L.OPT_RC_SKIP, 1)
    host = frames_host_ms(pts)
    print(json.dumps({"case": "svr_curve_frames 16384 stations (host)", "ms": round(host, 3)}), flush=True)
    print()
    print(f"{name}, {power}")
    print("| case | skip | ms | G taps/s | steps skipped | share of coherent ceiling |")
    print("|---|---|---|---|---|---|")
    for x in rows:
        skip = "-" if x["skip"] is None else ("on" if x["skip"] else "off")
        print(f"| {x['case']} | {skip} | {x['ms']:.3f} | {x['gtaps_per_s']:.1f} | {x['skipped_share']:.3f} | {x['share_of_coherent_ceiling']:.2f} |")
    print(f"| svr_curve_frames, 16384 stations (host) | - | {host:.3f} | | | |")
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump({"card": name, "power": power, "rows": rows, "curve_frames_host_ms": host}, f, indent=1)
    r.close()


if __name__ == "__main__":
    main()
