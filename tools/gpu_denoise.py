"""Denoising (svr_pathtracer_guides + svr_pathtracer_denoise) against raw sample means, C3 default and close view (camera at
0.45 x the framing distance, as bench.py).

Reference: a uniform render at 8192 spp (8 accumulate calls of 1024, samples disjoint from every row's).  Raw rows: uniform 64,
128, 256, 1024 spp.  Denoised rows: uniform 64, 128, 256 (rendered by svr_pathtracer_accumulate_adaptive with min = max, which
fills the odd-sample half the filter needs), and adaptive 2/255 (min 64, batch 64, max 1024) + denoise; filter defaults, guides
at 4 rays per pixel.  Per row: ms of the render, of the guide pass at 1, 4 and 16 rays per pixel and of the filter, each by CUDA
events (best of 3 after a warm-up); display-space RMSE against the reference and the fraction of pixels within 1/255 of it
(every channel).  Headline: the fastest denoised row at or below raw 256 spp's RMSE against raw 256 spp's time, with and without
the guide pass (guides are reused across renders of one view).  --sweep: the parameter grid behind svr_denoise_defaults, on
denoised 64 and 256 spp in both views.  Prints the card and its power limit; --json PATH also writes the rows as JSON."""
import argparse
import ctypes as C
import itertools
import json
import subprocess
import sys

import torch

sys.path.insert(0, ".")
from sunvolumerender_b200 import _lib as L  # noqa: E402
from sunvolumerender_b200 import scene as S  # noqa: E402
from sunvolumerender_b200.render import Renderer, setup_config  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return name, q.stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers below still stand; the power limit is then unknown
        return name, f"power limit unavailable ({e})"


def tone(x, exposure):
    return (1.0 - torch.exp(-x * 16.0 * exposure)) ** 2.2


def mean_of(sum_buf, H, W):
    v = sum_buf.view(H, W, 4)
    return v[..., :3] / v[..., 3:4].clamp_min(1.0)


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
    ap.add_argument("--sweep", action="store_true", help="also run the parameter grid behind the defaults")
    args = ap.parse_args()
    r = Renderer(0)
    cfg = S.CONFIGS["C3"]
    setup_config(r, cfg)
    name, power = card()
    print(f"card: {name}; power.limit, clocks.max.sm: {power}", flush=True)
    W, H = cfg.width, cfg.height
    npix = W * H
    depth = cfg.trace_depth
    buf = torch.zeros(npix * 4, dtype=torch.float32, device="cuda")
    half = torch.zeros_like(buf)
    ac = torch.zeros_like(buf)
    nd = torch.zeros_like(buf)
    cam0 = r.camera
    defaults = L.DenoiseParams()
    L.check(r.lib.svr_denoise_defaults(C.byref(defaults)), "svr_denoise_defaults")
    results = {"card": name, "power": power, "defaults": {f: getattr(defaults, f) for f, _ in L.DenoiseParams._fields_}, "views": {}}
    sweep_renders = {}
    for view in ("default", "close"):
        if view == "close":
            r.set_camera(S.make_camera((0, 0, cam0.pos.z * 0.45), (1, 0, 0), (0, 1, 0), (0, 0, 1), 45.0, 0.0, 1.0, 1.0, W, H))
        exposure = r.camera.exposure
        ref_buf = torch.zeros_like(buf)
        for b in range(8):
            r.accumulate(ref_buf, depth, (1 << 24) + b * 1024, 1024, clear=b == 0)
        torch.cuda.synchronize()
        ref = tone(mean_of(ref_buf, H, W), exposure)
        del ref_buf

        def quality(disp):
            d = disp - ref
            return float(d.square().mean().sqrt()), float((d.abs().amax(dim=-1) <= 1.0 / 255.0).float().mean())

        guide_ms = {k: timed(lambda k=k: r.guides(ac, nd, rays_per_pixel=k))[0] for k in (1, 4, 16)}
        r.guides(ac, nd, rays_per_pixel=4)

        def denoised(**kw):
            r.denoise(buf, half, (ac, nd), **kw)
            return tone(r.hdr.view(H, W, 3), exposure)

        rows = []
        for spp in (64, 128, 256, 1024):
            ms, _ = timed(lambda: r.accumulate(buf, depth, 0, spp, clear=True))
            e, within = quality(tone(mean_of(buf, H, W), exposure))
            rows.append({"kind": "raw", "spp": spp, "render_ms": ms, "samples": npix * spp, "rmse": e, "within_1_255": within})
        for spp in (64, 128, 256, None):
            if spp is None:
                ms, info = timed(lambda: r.accumulate_adaptive(buf, half, depth, 0, 64, 1024, 64, 2.0 / 255.0))
            else:
                ms, info = timed(lambda: r.accumulate_adaptive(buf, half, depth, 0, spp, spp, 32, 0.0))
            fms, _ = timed(lambda: r.denoise(buf, half, (ac, nd)))
            e, within = quality(denoised())
            row = {"kind": "denoised", "spp": spp, "adaptive_threshold_x255": None if spp else 2.0, "render_ms": ms, "samples": info["samples"],
                   "guides_ms": guide_ms, "filter_ms": fms, "rmse": e, "within_1_255": within}
            rows.append(row)
            if args.sweep and spp in (64, 256):
                sweep_renders[(view, spp)] = (buf.clone(), half.clone(), ac.clone(), nd.clone(), ref.clone(), exposure, r.camera)
        raw256 = next(x for x in rows if x["kind"] == "raw" and x["spp"] == 256)
        match = [x for x in rows if x["kind"] == "denoised" and x["rmse"] <= raw256["rmse"]]
        best = min(match, key=lambda x: x["render_ms"] + x["guides_ms"][4] + x["filter_ms"]) if match else None
        head = {"raw_256_ms": raw256["render_ms"], "raw_256_rmse": raw256["rmse"]}
        if best:
            head.update({"denoised_spp": best["spp"], "denoised_adaptive": best["spp"] is None, "with_guides_ms": best["render_ms"] + best["guides_ms"][4] + best["filter_ms"],
                         "without_guides_ms": best["render_ms"] + best["filter_ms"]})
        print(f"\n{view} view ({W} x {H}, reference 8192 spp); guides ms at 1 / 4 / 16 rays per pixel: "
              f"{guide_ms[1]:.3f} / {guide_ms[4]:.3f} / {guide_ms[16]:.3f}")
        print(f"{'row':>24} {'render ms':>10} {'filter ms':>10} {'spp/pixel':>10} {'RMSE':>10} {'<=1/255':>8}")
        for x in rows:
            label = f"raw {x['spp']}" if x["kind"] == "raw" else (f"denoised {x['spp']}" if x["spp"] else "adaptive 2/255 + denoise")
            f = f"{x['filter_ms']:10.3f}" if x["kind"] == "denoised" else f"{'':>10}"
            print(f"{label:>24} {x['render_ms']:10.2f} {f} {x['samples'] / npix:10.1f} {x['rmse']:10.6f} {x['within_1_255']:8.4f}")
        if best:
            label = f"denoised {best['spp']}" if best["spp"] else "adaptive 2/255 + denoise"
            print(f"headline: {label} reaches raw 256's RMSE ({raw256['rmse']:.6f}) in {head['with_guides_ms']:.2f} ms with 4-ray guides "
                  f"({head['without_guides_ms']:.2f} ms without) against {raw256['render_ms']:.2f} ms "
                  f"({raw256['render_ms'] / head['with_guides_ms']:.2f}x / {raw256['render_ms'] / head['without_guides_ms']:.2f}x)")
        else:
            print("headline: no denoised row reaches raw 256's RMSE")
        results["views"][view] = {"rows": rows, "headline": head}
    if args.sweep:
        grid = list(itertools.product((3, 4, 5), (2.0, 4.0, 8.0), (32.0, 128.0), (0.5, 1.0, 2.0, 4.0), (0.05, 0.1, 0.3)))
        sweep = []
        for it, sl, sn, sz, sa in grid:
            entry = {"iterations": it, "sigma_luminance": sl, "sigma_normal": sn, "sigma_depth": sz, "sigma_coverage": sa}
            for (view, spp), (b, h, a, n, ref, exposure, cam) in sweep_renders.items():
                r.set_camera(cam)
                r.denoise(b, h, (a, n), iterations=it, sigma_luminance=sl, sigma_normal=sn, sigma_depth=sz, sigma_coverage=sa)
                d = tone(r.hdr.view(H, W, 3), exposure) - ref
                entry[f"{view}_{spp}"] = float(d.square().mean().sqrt())
            sweep.append(entry)
        keys = [k for k in sweep[0] if k.endswith(("_64", "_256"))]
        base = {k: min(e[k] for e in sweep) for k in keys}
        for e in sweep:  # the mean over views and sample counts of RMSE / that column's best
            e["score"] = sum(e[k] / base[k] for k in keys) / len(keys)
        sweep.sort(key=lambda e: e["score"])
        print("\nsweep (RMSE per view and spp; score = mean of RMSE / the column's best), best 15 and the defaults:")
        dflt = (defaults.iterations, defaults.sigmaLuminance, defaults.sigmaNormal, defaults.sigmaDepth, round(defaults.sigmaCoverage, 6))
        for i, e in enumerate(sweep):
            is_default = (e["iterations"], e["sigma_luminance"], e["sigma_normal"], e["sigma_depth"], e["sigma_coverage"]) == dflt
            if i < 15 or is_default:
                cols = " ".join(f"{k} {e[k]:.6f}" for k in keys)
                print(f"{i + 1:4d} it {e['iterations']} sl {e['sigma_luminance']:g} sn {e['sigma_normal']:g} sz {e['sigma_depth']:g} sa {e['sigma_coverage']:g}: "
                      f"{cols} score {e['score']:.4f}{'  (defaults)' if is_default else ''}")
        results["sweep"] = sweep
    if args.json:
        with open(args.json, "w") as f:
            json.dump(results, f, indent=1)
    r.close()


if __name__ == "__main__":
    main()
