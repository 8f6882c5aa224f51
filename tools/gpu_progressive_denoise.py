"""The denoised progressive display (SVR_OPT_PT_DENOISE) on C3, default and close view (camera at 0.45 x the framing distance,
as bench.py): what a user of render_pathtracer -- the reference GUI, the canvas -- sees frame by frame with the option off and on.

Per view:
  * steady state: ms per render_pathtracer frame over frames 20..275 (CUDA events around the 256 calls): option off (look-ahead
    as by default), option off with look-ahead off (the plain one-sample trace and tone map), option on (4 rays); the filter
    alone (svr_pathtracer_denoise at the same size, 256 calls) -- trace = on - filter;
  * first frame after setup_camera + frameNo = 0: off, and on with 1, 4 and 16 guide rays (best of 6);
  * the frame-16 refinement: frames 14..17 of a 4-ray render timed one by one; cost = frame 16 - mean of frames 15 and 17;
  * display RMSE and the share of pixels within 1/255 (every channel) of the u8 image shown after 1, 2, 4, ..., 256 and 1024
    frames, raw (option off: the running mean's tone map) against denoised (option 4), against the u8 image of an 8192-spp
    render (8 accumulate calls of 1024, samples disjoint from the render's; tone-mapped and truncated to u8 as every image is);
  * the first frame at which each reaches raw frame 256's RMSE, and the wall time of that many frames from a restart (CUDA
    events around the whole run, guide passes included).
Prints the card and its power limit; --json PATH also writes the results."""
import argparse
import ctypes as C
import json
import subprocess
import sys

import torch

sys.path.insert(0, ".")
from sunvolumerender_b200 import _lib as L  # noqa: E402
from sunvolumerender_b200 import scene as S  # noqa: E402
from sunvolumerender_b200.render import Renderer, setup_config  # noqa: E402

MARKS = (1, 2, 4, 8, 16, 32, 64, 128, 256, 1024)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return name, q.stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers below still stand; the power limit is then unknown
        return name, f"power limit unavailable ({e})"


class Frames:
    def __init__(self, r, depth):
        self.r, self.depth = r, depth
        self.rp = L.RenderParams(depth, 0, r.hdr.data_ptr())
        self.img = C.c_void_p(r.img.data_ptr())

    def __call__(self, f):
        self.rp.frameNo = f
        self.r.lib.render_pathtracer(self.img, C.byref(self.rp))


def events(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json", default=None, help="write the results to this file")
    args = ap.parse_args()
    r = Renderer(0)
    cfg = S.CONFIGS["C3"]
    setup_config(r, cfg)
    name, power = card()
    print(f"card: {name}; power.limit, clocks.max.sm: {power}", flush=True)
    W, H, depth = cfg.width, cfg.height, cfg.trace_depth
    npix = W * H
    frame = Frames(r, depth)
    cam0 = r.camera
    lookahead = r.get_option(L.OPT_PT_LOOKAHEAD)
    results = {"card": name, "power": power, "views": {}}
    for view in ("default", "close"):
        cam = cam0 if view == "default" else S.make_camera((0, 0, cam0.pos.z * 0.45), (1, 0, 0), (0, 1, 0), (0, 0, 1), 45.0, 0.0, 1.0, 1.0, W, H)
        r.set_camera(cam)
        ex = cam.exposure
        ref_buf = torch.zeros(npix * 4, dtype=torch.float32, device="cuda")
        for b in range(8):
            r.accumulate(ref_buf, depth, (1 << 24) + b * 1024, 1024, clear=b == 0)
        v = ref_buf.view(H, W, 4)
        ref = torch.floor(((1.0 - torch.exp(-(v[..., :3] / v[..., 3:4]) * 16.0 * ex)) ** 2.2) * 255.0) / 255.0  # as pack_u8x4 truncates
        del ref_buf, v

        def restart(value, la=lookahead):
            r.set_option(L.OPT_PT_DENOISE, value)
            r.set_option(L.OPT_PT_LOOKAHEAD, la)
            r.lib.setup_camera(C.byref(cam))

        # ---- steady state, frames 20..275
        steady = {}
        for label, value, la in (("off", 0, lookahead), ("off_no_lookahead", 0, 0), ("on", 4, lookahead)):
            restart(value, la)
            for f in range(20):
                frame(f)
            torch.cuda.synchronize()
            steady[label] = events(lambda: [frame(f) for f in range(20, 276)]) / 256.0
        restart(0)
        s = torch.zeros(npix * 4, dtype=torch.float32, device="cuda")
        half, ac, nd = torch.zeros_like(s), torch.zeros_like(s), torch.zeros_like(s)
        r.accumulate(s, depth, 0, 64, clear=True)
        r.accumulate(half, depth, 64, 32, clear=True)
        r.guides(ac, nd, rays_per_pixel=4)
        ptrs = [C.c_void_p(t.data_ptr()) for t in (s, half, ac, nd)]
        img = C.c_void_p(r.img.data_ptr())
        r.lib.svr_pathtracer_denoise(img, None, *ptrs, None)
        torch.cuda.synchronize()
        steady["filter"] = events(lambda: [r.lib.svr_pathtracer_denoise(img, None, *ptrs, None) for _ in range(256)]) / 256.0
        steady["trace_on"] = steady["on"] - steady["filter"]
        del s, half, ac, nd

        # ---- first frame after a camera change
        first = {}
        for label, value in (("off", 0), ("on_1", 1), ("on_4", 4), ("on_16", 16)):
            best = 1e30
            for _ in range(6):
                restart(value)
                best = min(best, events(lambda: frame(0)))
                for f in range(1, 3):
                    frame(f)
            first[label] = best

        # ---- the frame-16 refinement (4-ray guides remade at 16 rays)
        per = {}
        for rep in range(3):
            restart(4)
            for f in range(14):
                frame(f)
            for f in range(14, 18):
                t = events(lambda f=f: frame(f))
                per[f] = min(per.get(f, 1e30), t)
        refine = per[16] - 0.5 * (per[15] + per[17])

        # ---- quality, frame by frame
        def quality():
            d = r.img.view(H, W, 4)[..., :3].float() / 255.0 - ref
            return float(d.square().mean().sqrt()), float((d.abs().amax(dim=-1) <= 1.0 / 255.0 + 1e-6).float().mean())

        curve = {}
        for label, value in (("raw", 0), ("denoised", 4)):
            restart(value)
            curve[label] = []
            for f in range(max(MARKS)):
                frame(f)
                curve[label].append(quality())
        target = curve["raw"][255][0]
        reach = {}
        for label, value in (("raw", 0), ("denoised", 4)):
            n = next((i + 1 for i, (e, _) in enumerate(curve[label]) if e <= target), None)
            if n is None:
                reach[label] = None
                continue
            restart(value)
            torch.cuda.synchronize()
            reach[label] = {"frames": n, "ms": events(lambda n=n: [frame(f) for f in range(n)])}
        restart(0)
        results["views"][view] = {"steady_ms": steady, "first_frame_ms": first, "frames_14_17_ms": per, "refine_ms": refine,
                                  "quality": {lab: {n: curve[lab][n - 1] for n in MARKS} for lab in curve}, "reach_raw_256": reach}

        print(f"\n{view} view ({W} x {H}, depth {depth}; reference 8192 spp)")
        print("ms per frame, frames 20..275: off {off:.3f} (look-ahead off: {off_no_lookahead:.3f}); on {on:.3f} = trace {trace_on:.3f} + filter "
              "{filter:.3f}".format(**steady))
        print("first frame after setup_camera, ms: off {off:.3f}; on, 1 / 4 / 16 rays: {on_1:.3f} / {on_4:.3f} / {on_16:.3f}".format(**first))
        print("frames 14..17, ms: " + " ".join(f"{per[f]:.3f}" for f in range(14, 18)) + f"; frame-16 refinement costs {refine:.3f} ms")
        print(f"{'frames':>7} {'raw RMSE':>10} {'den. RMSE':>10} {'ratio':>6} {'raw <=1/255':>12} {'den. <=1/255':>12}")
        for n in MARKS:
            (e0, w0), (e1, w1) = curve["raw"][n - 1], curve["denoised"][n - 1]
            print(f"{n:7d} {e0:10.6f} {e1:10.6f} {e1 / e0:6.3f} {w0:12.4f} {w1:12.4f}")
        for label in ("raw", "denoised"):
            x = reach[label]
            print(f"{label} reaches raw 256's RMSE ({target:.6f}): " + (f"frame {x['frames']}, {x['ms']:.2f} ms from a restart" if x else "not within 1024 frames"))
    r.set_option(L.OPT_PT_DENOISE, 0)
    if args.json:
        with open(args.json, "w") as f:
            json.dump(results, f, indent=1)
    r.close()


if __name__ == "__main__":
    main()
