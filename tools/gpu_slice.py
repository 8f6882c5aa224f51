"""Slices and slabs (svr_render_slices) on C3 (512^3 u16 CT, 256 MB of voxels: more than the 126 MB L2):
  * a thin 1024 x 1024 axial and oblique slice (half a voxel per pixel): one fetch per pixel, launch-bound;
  * a 512-slice stack of 512 x 512 slices, axial and oblique (one voxel per pixel and per slice): the reformat, 134 M fetches;
  * 64-sample MIP, MinIP and AIP slabs (64 voxels thick, one sample per voxel) at 1024 x 1024, axial and oblique, with
    skipping (SVR_OPT_RC_SKIP) on and off; the value and image are checked equal with torch.equal.
Per row: ms per call (CUDA events around 10 calls, best of 5 windows after a warm-up), G taps/s (executed taps from a separate
counters run, over the timed call), the share of steps skipped, and taps/s as a share of the coherent tex3D ceiling on the
same volume (svr_microbench_taps, as tools/gpu_projection.py).  Prints the card and its power limit, then a markdown table;
--json PATH also writes the results."""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sunvolumerender_b200 import _lib as L  # noqa: E402
from sunvolumerender_b200 import scene as S  # noqa: E402
from sunvolumerender_b200.render import Renderer, setup_config  # noqa: E402

from gpu_projection import card, coherent_ceiling, counted, events  # noqa: E402

OBLIQUE = ((0.3, 0.2, 1.0), (0.0, 1.0, 0.0))  # normal, up


def cases(n):
    dims, sp = (n, n, n), (1.0, 1.0, 1.0)

    def axial(size, count=1, slab=0, mode="max"):
        p = S.axis_slice(dims, sp, "z", n // 2 if count == 1 else 0, thickness_voxels=slab, count=count, mode=mode)
        p.imageW = p.imageH = size
        p.axisU[0] = p.axisV[1] = n / size
        return p

    def oblique(size, count=1, slab=0, mode="max"):
        normal, up = OBLIQUE
        u = torch.tensor(normal, dtype=torch.float64)
        u = u / u.norm()
        c = (-(count - 1) / 2.0 * u).tolist()  # the stack is centred on the volume's centre
        return S.oblique_slice(c, normal, up, n / size, size, size, count=count, slice_step=1.0, thickness=float(slab), sample_spacing=1.0,
                               mode=mode)

    out = [("thin 1024^2", "axial", axial(1024)), ("thin 1024^2", "oblique", oblique(1024)),
           ("stack 512 x 512^2", "axial", axial(512, count=512)), ("stack 512 x 512^2", "oblique", oblique(512, count=512))]
    for mode in ("max", "min", "mean"):
        out += [(f"slab 64 {mode}", "axial", axial(1024, slab=64, mode=mode)), (f"slab 64 {mode}", "oblique", oblique(1024, slab=64, mode=mode))]
    return out


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
    rows = []
    for what, view, p in cases(cfg.n):
        shape = (p.count, p.imageH, p.imageW)
        value = torch.empty(shape, dtype=torch.float32, device="cuda")
        img = torch.empty(shape + (4,), dtype=torch.uint8, device="cuda")
        outs = {}
        for skip in ((1, 0) if p.thickness > 0 else (1,)):
            r.set_option(L.OPT_RC_SKIP, skip)
            fn = lambda: r.render_slices(p, value, img)  # noqa: E731
            ms = events(fn)
            c = counted(r, fn)
            outs[skip] = (value.clone(), img.clone())
            gtaps = c["shade_taps"] / (ms * 1e-3) / 1e9
            row = {"case": what, "view": view, "skip": skip if p.thickness > 0 else None, "ms": round(ms, 4), "pixels": c["paths"],
                   "gtaps_per_s": round(gtaps, 2), "skipped_share": round(c["skipped"] / max(c["steps"], 1), 4), "steps": c["steps"],
                   "share_of_coherent_ceiling": round(gtaps / ceiling, 3), "coherent_ceiling_gtaps_per_s": round(ceiling, 1)}
            rows.append(row)
            print(json.dumps(row), flush=True)
        if len(outs) == 2:
            assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]), (what, view)
        del value, img, outs
    r.set_option(L.OPT_RC_SKIP, 1)
    print()
    print(f"{name}, {power}")
    print("| case | view | skip | ms | G taps/s | steps skipped | share of coherent ceiling |")
    print("|---|---|---|---|---|---|---|")
    for x in rows:
        skip = "-" if x["skip"] is None else ("on" if x["skip"] else "off")
        print(f"| {x['case']} | {x['view']} | {skip} | {x['ms']:.3f} | {x['gtaps_per_s']:.1f} | {x['skipped_share']:.3f} | "
              f"{x['share_of_coherent_ceiling']:.2f} |")
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump({"card": name, "power": power, "rows": rows}, f, indent=1)
    r.close()


if __name__ == "__main__":
    main()
