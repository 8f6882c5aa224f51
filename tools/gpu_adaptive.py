"""Adaptive sampling against uniform sampling, C3 default and close view (camera at 0.45 x the framing distance, as bench.py).

Reference: a uniform render at 8192 spp (8 accumulate calls of 1024, samples disjoint from every row's).  Rows: uniform 64 .. 1024
spp, adaptive at thresholds 2, 1, 0.5 / 255 (min 64, batch 64, max 1024).  Per row: ms by CUDA events (best of 3; an adaptive
render's per-round synchronisations included), samples traced, rounds, display-space RMSE against the reference and the fraction
of pixels within 1/255 of it (every channel).  Headline: the fastest adaptive row at or below the RMSE of uniform 256 spp, against
uniform 256 spp.  Prints the card and its power limit; --json PATH also writes the rows as JSON."""
import argparse
import json
import subprocess
import sys

import torch

sys.path.insert(0, ".")
from sunvolumerender_b200 import scene as S  # noqa: E402
from sunvolumerender_b200.render import Renderer, setup_config  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return name, q.stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers below still stand; the power limit is then unknown
        return name, f"power limit unavailable ({e})"


def display(sum_buf, exposure, H, W):
    v = sum_buf.view(H, W, 4)
    L = v[..., :3] / v[..., 3:4].clamp_min(1.0)
    return (1.0 - torch.exp(-L * 16.0 * exposure)) ** 2.2


def timed(fn, reps=3):
    best, out = 1e30, None
    fn()  # warm-up
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json", default=None, help="write the rows and headlines to this file")
    args = ap.parse_args()
    r = Renderer(0)
    cfg = S.CONFIGS["C3"]
    setup_config(r, cfg)
    name, power = card()
    print(f"card: {name}; power.limit, clocks.max.sm: {power}", flush=True)
    W, H = cfg.width, cfg.height
    npix = W * H
    buf = torch.zeros(npix * 4, dtype=torch.float32, device="cuda")
    half = torch.zeros_like(buf)
    cam0 = r.camera
    results = {"card": name, "power": power, "views": {}}
    for view in ("default", "close"):
        if view == "close":
            r.set_camera(S.make_camera((0, 0, cam0.pos.z * 0.45), (1, 0, 0), (0, 1, 0), (0, 0, 1), 45.0, 0.0, 1.0, 1.0, W, H))
        exposure = r.camera.exposure
        ref_buf = torch.zeros_like(buf)
        for b in range(8):
            r.accumulate(ref_buf, cfg.trace_depth, (1 << 24) + b * 1024, 1024, clear=b == 0)
        torch.cuda.synchronize()
        ref = display(ref_buf, exposure, H, W)
        del ref_buf

        def quality():
            d = display(buf, exposure, H, W) - ref
            return float(d.square().mean().sqrt()), float((d.abs().amax(dim=-1) <= 1.0 / 255.0).float().mean())

        rows = []
        for spp in (64, 128, 256, 512, 1024):
            ms, _ = timed(lambda: r.accumulate(buf, cfg.trace_depth, 0, spp, clear=True))
            e, within = quality()
            rows.append({"kind": "uniform", "spp": spp, "ms": ms, "samples": npix * spp, "rounds": 1, "rmse": e, "within_1_255": within})
        for t in (2.0, 1.0, 0.5):
            ms, info = timed(lambda: r.accumulate_adaptive(buf, half, cfg.trace_depth, 0, 64, 1024, 64, t / 255.0))
            e, within = quality()
            rows.append({"kind": "adaptive", "threshold_x255": t, "ms": ms, "samples": info["samples"], "rounds": info["rounds"],
                         "unconverged": info["unconverged"], "rmse": e, "within_1_255": within})
        u256 = next(x for x in rows if x["kind"] == "uniform" and x["spp"] == 256)
        match = [x for x in rows if x["kind"] == "adaptive" and x["rmse"] <= u256["rmse"]]
        best = min(match, key=lambda x: x["ms"]) if match else None
        head = {"uniform_256_ms": u256["ms"], "uniform_256_rmse": u256["rmse"],
                "adaptive_ms": best["ms"] if best else None, "adaptive_threshold_x255": best["threshold_x255"] if best else None}
        print(f"\n{view} view ({W} x {H}, reference 8192 spp)")
        print(f"{'row':>18} {'ms':>9} {'spp/pixel':>10} {'rounds':>7} {'RMSE':>10} {'<=1/255':>8}")
        for x in rows:
            label = f"uniform {x['spp']}" if x["kind"] == "uniform" else f"adaptive {x['threshold_x255']:g}/255"
            print(f"{label:>18} {x['ms']:9.2f} {x['samples'] / npix:10.1f} {x['rounds']:7d} {x['rmse']:10.6f} {x['within_1_255']:8.4f}")
        if best:
            print(f"headline: adaptive {best['threshold_x255']:g}/255 reaches uniform 256's RMSE ({u256['rmse']:.6f}) in {best['ms']:.2f} ms "
                  f"against {u256['ms']:.2f} ms ({u256['ms'] / best['ms']:.2f}x)")
        else:
            print("headline: no adaptive row reaches uniform 256's RMSE")
        results["views"][view] = {"rows": rows, "headline": head}
    if args.json:
        with open(args.json, "w") as f:
            json.dump(results, f, indent=1)
    r.close()


if __name__ == "__main__":
    main()
