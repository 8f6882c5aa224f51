"""Label maps on C3 (512^3 u16 CT): skin (1), soft tissue (2) and bone (3) from scene.labels_from_thresholds at
scene.CT_LABEL_LEVELS, on the CT's grid.

3D (svr_render_labels), 1920 x 1080, the default view and the close view (camera at 0.45 x the framing distance, as
tools/gpu_isosurface.py), with two tables (all three labels visible; bone alone) and skipping on and off (SVR_OPT_RC_SKIP):
  * ms per frame: CUDA events around 10 frames, best of 5 windows after a warm-up;
  * from a separate counters run (SVR_OPT_COUNTERS): the share of steps skipped, indicator evaluations per ray, hits;
  * render_isosurface at 0.7 on the same frame (both are first-hit renderers), skipping on;
  * a check that img, surface and label are torch.equal with skipping on and off.
Overlays (svr_render_label_slices) on C3: a thin 1024^2 axial slice through the centre (0.5 voxel pixels) without and with
outline, next to the grey svr_render_slices call it goes over, and a 512-slice axial stack at 512^2 (labels and composite).
Prints the card and its power limit, then markdown tables; --json PATH also writes the results."""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sunvolumerender_b200 import _lib as L  # noqa: E402
from sunvolumerender_b200 import scene as S  # noqa: E402
from sunvolumerender_b200.render import Renderer, setup_config  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from gpu_projection import card, counted, events  # noqa: E402

TABLES = {"all": S.label_table(S.label_palette(3)), "bone": S.label_table({3: (1.0, 1.0, 0.9, 1.0)})}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    name, power = card()
    print(f"card: {name}; power.limit, clocks.max.sm: {power}", flush=True)
    r = Renderer(0)
    cfg = S.CONFIGS["C3"]
    vox = setup_config(r, cfg)
    n = cfg.n
    labels = S.labels_from_thresholds(vox.cpu().numpy().view(S.VOXEL_DTYPES[cfg.fmt]).reshape(n, n, n), S.CT_LABEL_LEVELS)
    del vox
    r.load_labels(labels)
    del labels
    r.set_option(L.OPT_MACROCELL_SIZE, 0)
    step = S.raycast_step_size(r.volume.spacing.tuple())
    W, H = cfg.width, cfg.height
    surface = torch.empty(W * H * 4, dtype=torch.float32, device="cuda")
    lab = torch.empty(W * H, dtype=torch.uint8, device="cuda")
    base = S.default_camera(cfg.extent, W, H)
    rows3d = []
    for view in ("default", "close"):
        cam = base if view == "default" else S.make_camera((0.0, 0.0, 0.45 * base.pos.z), (1, 0, 0), (0, 1, 0), (0, 0, 1), 45.0, 0.0, 1.0, 1.0, W, H)
        r.set_camera(cam)
        r.set_option(L.OPT_RC_SKIP, 1)
        iso_ms = events(lambda: r.render_isosurface(0.7, step))
        for tname, table in TABLES.items():
            outputs = {}
            for skip in (1, 0):
                r.set_option(L.OPT_RC_SKIP, skip)
                fn = lambda: r.render_labels(table, step, surface=surface, labels=lab)  # noqa: E731
                ms = events(fn)
                c = counted(r, fn)
                outputs[skip] = (r.img.clone(), surface.clone(), lab.clone())
                hits = int(torch.isfinite(surface.view(-1, 4)[:, 3]).sum())
                row = {"view": view, "table": tname, "skip": skip, "ms": round(ms, 4), "skipped_share": round(c["skipped"] / max(c["steps"], 1), 4),
                       "evals_per_ray": round(c["shade_taps"] / max(c["paths"], 1), 1), "hit_share": round(hits / max(c["paths"], 1), 4),
                       "iso07_ms": round(iso_ms, 4)}
                rows3d.append(row)
                print(json.dumps(row), flush=True)
            same = all(torch.equal(a, b) for a, b in zip(outputs[0], outputs[1]))
            rows3d[-1]["equal"] = rows3d[-2]["equal"] = same
            assert same, (view, tname)
    r.set_option(L.OPT_RC_SKIP, 1)
    # overlays
    rows2d = []
    thin = S.oblique_slice((0.0, 0.0, 0.0), (0.0, 0.0, 1.0), (0.0, 1.0, 0.0), 0.5, 1024, 1024)
    value, img = r.render_slices(thin)
    labels2d = torch.empty((1, 1024, 1024), dtype=torch.uint8, device="cuda")
    grey_ms = events(lambda: r.render_slices(thin, value, img), frames=50)
    for outline in (False, True):
        ms = events(lambda: r.render_label_slices(thin, TABLES["all"], img=img, labels=labels2d, outline=outline), frames=50)
        rows2d.append({"case": "thin 1024^2 axial", "outline": outline, "ms": round(ms, 4), "grey_slice_ms": round(grey_ms, 4)})
        print(json.dumps(rows2d[-1]), flush=True)
    stack = S.axis_slice((n, n, n), (1.0, 1.0, 1.0), "z", 0, count=n)
    value, img = r.render_slices(stack)
    labels3 = torch.empty((n, n, n), dtype=torch.uint8, device="cuda")
    grey_ms = events(lambda: r.render_slices(stack, value, img), frames=5)
    for outline in (False, True):
        ms = events(lambda: r.render_label_slices(stack, TABLES["all"], img=img, labels=labels3, outline=outline), frames=5)
        rows2d.append({"case": "512-slice stack of 512^2", "outline": outline, "ms": round(ms, 4), "grey_slice_ms": round(grey_ms, 4)})
        print(json.dumps(rows2d[-1]), flush=True)
    print()
    print(f"{name}, {power}")
    print("| view | table | skip | ms | steps skipped | indicator evaluations per ray | hits | render_isosurface 0.7 ms | equal on/off |")
    print("|---|---|---|---|---|---|---|---|---|")
    for x in rows3d:
        print(f"| {x['view']} | {x['table']} | {'on' if x['skip'] else 'off'} | {x['ms']:.3f} | {x['skipped_share']:.3f} | {x['evals_per_ray']:.1f} | "
              f"{x['hit_share']:.3f} | {x['iso07_ms']:.3f} | {x['equal']} |")
    print()
    print("| overlay | outline | ms | grey svr_render_slices ms |")
    print("|---|---|---|---|")
    for x in rows2d:
        print(f"| {x['case']} | {'on' if x['outline'] else 'off'} | {x['ms']:.4f} | {x['grey_slice_ms']:.4f} |")
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump({"card": name, "power": power, "surfaces": rows3d, "overlays": rows2d}, f, indent=1)
    r.close()


if __name__ == "__main__":
    main()
