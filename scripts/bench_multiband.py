"""Measurement of the multi-band blend (include/mcs.h mcs_plan_set_multiband) on one GPU.

Inputs resident in HBM, two batches of distinct frame-sets alternated so that every launch reads fresh
inputs, CUDA events around the timed launches after a warm-up.  Per workload (config 2 = 6 x 1080p and
ns_8x1080p = 8 x 1080p, BGR, edge ramps of 64 px as masks) and per frame count F (16 and 64 per launch)
four legs, alternated round by round:
  mb3, mb5     the multi-band blend at 3 and 5 bands (variant 6)
  cw           the single-band camera-weighted blend of the same masks (variant 5)
  overwrite    the reference's overwrite (tiled kernel)
Before timing, frame 0 of each multi-band leg is compared with oracle/multiband_model.blend.  The CPU
baseline times cv2.detail_MultiBandBlender (prepare, feed, blend; OpenCV's own threads) on frame-set 0
with the planes precomputed.  The intermediate bytes per panorama are computed from the feed regions:
each kernel's int16 reads and writes of the camera and panorama pyramids, weights and weight sums, each
element counted once per kernel that touches it (plus the source samples and the u8 output).

    python scripts/bench_multiband.py [--launches 10] [--rounds 3] [--out profiles/multiband.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {"cfg2_6x1080p": (6, 1080, 1920), "ns_8x1080p": (8, 1080, 1920)}
FRAMES = (16, 64)
DISTINCT = 4


def gpu_info(torch):
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [v.strip() for v in q.split(",")[:2]]
    except Exception as e:
        info["power_limit"] = "unknown (%s)" % e
    return info


def intermediate_bytes(planes, out_w, out_h, bands, C):
    """int16 bytes the pipeline reads and writes per panorama, from the feed regions (module docstring)."""
    from oracle import multiband_model as mb
    n = mb.num_bands(bands, out_w, out_h)
    RW, RH = mb.roi_size(n, out_w, out_h)
    regions = [mb.feed_region(r, n, RW, RH) for r, _, _ in planes]
    cam = [[((b[2] - b[0]) >> i) * ((b[3] - b[1]) >> i) for i in range(n + 1)] for b in regions]
    pan = [(RW >> i) * (RH >> i) for i in range(n + 1)]
    total = 0
    for px in cam:
        total += px[0] * C * (1 + 2)                                   # level 0: source taps (u8, ~1 each) + int16 store
        for i in range(n):
            total += (px[i] + px[i + 1]) * C * 2                       # pyrDown: read level i, write level i + 1
        for i in range(n + 1):
            total += (px[i] * C + (px[i + 1] * C if i < n else 0)) * 2 + px[i] * 2   # blend: G_i, G_i+1, weights
    for i in range(n + 1):
        total += pan[i] * 2                                            # weight sums
        total += (pan[i + 1] * C * 2 if i < n else 0)                  # collapse: restored level i + 1
        total += pan[i] * C * 2 if i > 0 else out_w * out_h * C        # store level i (level 0: u8 output)
    return int(total)


def run_workload(torch, name, launches, rounds):
    import cv2
    from multicamera_stitching_b200 import edge_ramp, synthetic
    from multicamera_stitching_b200.plan import flatten_chain
    from oracle import multiband_model as mb
    dev = torch.device("cuda", 0)
    n, h, w = WORKLOADS[name]
    st, _, labels, images = synthetic.synthetic_stitcher(n, h, w, 3, kind="smooth")
    shapes = [images[l].shape for l in labels]
    maps = {l: edge_ramp(images[l].shape, 64) for l in labels}
    flat = flatten_chain(st.stitchers, shapes)
    host_sets = [images] + [synthetic.make_frames(n, h, w, 3, f, "smooth") for f in range(1, DISTINCT)]
    B = max(FRAMES)
    xor = torch.arange(2 * B, dtype=torch.uint8, device=dev).view(-1, 1, 1, 1)
    frames = {}
    for l in labels:
        base = torch.from_numpy(np.stack([s[l] for s in host_sets])).to(dev)
        frames[l] = base[torch.arange(2 * B, device=dev) % DISTINCT] ^ xor
    batches = [{l: frames[l][b * B:(b + 1) * B] for l in labels} for b in range(2)]

    legs = {}
    for leg, cw, bands in (("mb3", maps, 3), ("mb5", maps, 5), ("cw", maps, 0), ("overwrite", None, 0)):
        st.camera_weights, st.blend_bands = cw, bands
        plan = st.plan(shapes, dev)
        legs[leg] = dict(plan=plan, out=plan.new_output(B), bands=bands)
    st.camera_weights, st.blend_bands = None, 0

    def launch(leg, b, F):
        L = legs[leg]
        L["plan"].run([batches[b][l][:F] for l in labels], out=L["out"][:F], n_frames=F)

    frames0 = [images[l] for l in labels]
    planes = mb.camera_planes(flat.layers, flat.out_w, flat.out_h, frames0, [maps[l] for l in labels])
    checks, cpu = {}, {}
    for leg in ("mb3", "mb5"):
        launch(leg, 0, 1)
        torch.cuda.synchronize()
        ref = mb.blend(flat.layers, flat.out_w, flat.out_h, frames0, [maps[l] for l in labels], legs[leg]["bands"])
        checks[leg] = bool(np.array_equal(legs[leg]["out"][0].cpu().numpy(), ref))
        if not checks[leg]:
            raise SystemExit("%s %s: frame 0 differs from oracle/multiband_model.blend" % (name, leg))
        reps = []
        for _ in range(3):
            t0 = time.perf_counter()
            mb.cv2_blend3(planes, flat.out_w, flat.out_h, legs[leg]["bands"])
            reps.append(time.perf_counter() - t0)
        cpu[leg] = dict(seconds_best=round(min(reps), 4), panoramas_per_s=round(1.0 / min(reps), 2),
                        threads=cv2.getNumThreads())
    res = {}
    for F in FRAMES:
        for leg in legs:
            for b in (0, 1, 0, 1):
                launch(leg, b, F)
        torch.cuda.synchronize()
        ms = {leg: [] for leg in legs}
        variant = {}
        for _ in range(rounds):
            for leg in legs:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(launches):
                    launch(leg, i & 1, F)
                e1.record()
                torch.cuda.synchronize()
                ms[leg].append(e0.elapsed_time(e1) / launches)
                variant[leg] = legs[leg]["plan"].handle.last_variant()
        for leg in legs:
            best = min(ms[leg])
            r = dict(variant=variant[leg], ms_per_launch=[round(v, 4) for v in ms[leg]], ms_best=round(best, 4),
                     panoramas_per_s=round(F / best * 1e3, 1))
            if leg.startswith("mb"):
                ib = intermediate_bytes(planes, flat.out_w, flat.out_h, legs[leg]["bands"], 3)
                r.update(effective_bands=legs[leg]["plan"].handle.blend_bands, intermediate_bytes_per_panorama=ib,
                         intermediate_gbs=round(ib * F / best / 1e6, 1), frame0_equals_model=checks[leg],
                         cpu_cv2=cpu[leg])
            res["F%d_%s" % (F, leg)] = r
    return dict(workload=name, cameras=n, frame_hw=[h, w], panorama_hw=[flat.out_h, flat.out_w],
                launches_per_round=launches, rounds=rounds, legs=res)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", default="cfg2_6x1080p,ns_8x1080p")
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON record here")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_multiband.py needs a CUDA device")
    torch.cuda.set_device(0)
    rec = dict(bench="multiband", **gpu_info(torch),
               results=[run_workload(torch, w, args.launches, args.rounds) for w in args.workloads.split(",")])
    text = json.dumps(rec, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
