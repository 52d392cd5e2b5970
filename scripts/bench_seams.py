"""Measurement of the Voronoi seams of the multi-band blend (include/mcs.h mcs_plan_set_voronoi_seams) on one GPU.

Per workload (config 2 = 6 x 1080p and ns_8x1080p = 8 x 1080p, BGR, edge ramps of 64 px as masks, 5 bands):
  plan time    mcs_plan_set_voronoi_seams(plan, 1) (sample the weights, find the seams, rebuild the weight
               pyramids and sums) and (plan, 0) (the rebuild alone), host clock around the synchronous call,
               alternated; against oracle/seam_model.find_cv2 (cv2's VoronoiSeamFinder on OpenCV's own threads)
               on the same masks.  The read-back seam weights of every layer are compared with find_cv2 first.
  per frame    the multi-band blend with and without seams, inputs resident in HBM, F = 16 and 64 panoramas per
               launch, legs alternated round by round, CUDA events.  Frame 0 of the seams leg is compared with
               oracle/seam_model.blend_cv2 first.

    python scripts/bench_seams.py [--launches 10] [--rounds 3] [--reps 5] [--out profiles/seams.json]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402

from bench_multiband import DISTINCT, gpu_info  # noqa: E402

WORKLOADS = {"cfg2_6x1080p": (6, 1080, 1920), "ns_8x1080p": (8, 1080, 1920)}
FRAMES = (16, 64)
BANDS = 5


def run_workload(torch, name, launches, rounds, reps):
    import cv2
    from multicamera_stitching_b200 import edge_ramp, synthetic
    from multicamera_stitching_b200.plan import flatten_chain
    from oracle import multiband_model as mb
    from oracle import seam_model
    dev = torch.device("cuda", 0)
    n, h, w = WORKLOADS[name]
    st, _, labels, images = synthetic.synthetic_stitcher(n, h, w, 3, kind="smooth")
    shapes = [images[l].shape for l in labels]
    maps = {l: edge_ramp(images[l].shape, 64) for l in labels}
    flat = flatten_chain(st.stitchers, shapes)
    frames0, m = [images[l] for l in labels], [maps[l] for l in labels]
    planes = mb.camera_planes(flat.layers, flat.out_w, flat.out_h, frames0, m)
    sizes, corners, masks = seam_model.plane_inputs(planes)
    pairs = seam_model.find(sizes, corners, [np.zeros_like(k) for k in masks], details=True)[1]

    legs = {}
    for leg, seams in (("seams", True), ("no_seams", False)):
        st.camera_weights, st.blend_bands, st.voronoi_seams = maps, BANDS, seams
        plan = st.plan(shapes, dev)
        legs[leg] = dict(plan=plan, out=plan.new_output(max(FRAMES)))
    st.camera_weights, st.blend_bands, st.voronoi_seams = None, 0, False
    handle = legs["seams"]["plan"].handle

    # plan time: the read-back equals cv2's finder, then the calls timed, alternated
    ref = seam_model.find_cv2(sizes, corners, masks)
    fed = [k for k, l in enumerate(flat.layers) if handle.rects[k][2] > handle.rects[k][0] and handle.rects[k][3] > handle.rects[k][1]]
    seams_equal = all(np.array_equal(handle.seam_weights(k), r) for k, r in zip(fed, ref))
    if not seams_equal:
        raise SystemExit("%s: the seam weights differ from cv2's VoronoiSeamFinder" % name)
    on, off = [], []
    for _ in range(reps):
        for enable, acc in ((False, off), (True, on)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            handle.set_voronoi_seams(enable)
            acc.append((time.perf_counter() - t0) * 1e3)
    assert handle.voronoi_seams
    cpu = []
    for _ in range(reps):
        t0 = time.perf_counter()
        seam_model.find_cv2(sizes, corners, masks)
        cpu.append((time.perf_counter() - t0) * 1e3)
    plan_time = dict(pairs=len(pairs), launches=1 + 2 * len(pairs),
                     largest_submask_wh=max(seam_model.submask_size(r) for _, _, r in pairs),
                     seams_on_ms=[round(v, 2) for v in on], seams_on_ms_best=round(min(on), 2),
                     seams_off_ms=[round(v, 2) for v in off], seams_off_ms_best=round(min(off), 2),
                     cpu_cv2_find_ms=[round(v, 2) for v in cpu], cpu_cv2_find_ms_best=round(min(cpu), 2),
                     cpu_threads=cv2.getNumThreads(), seam_weights_equal_cv2=seams_equal)

    # per frame
    host_sets = [images] + [synthetic.make_frames(n, h, w, 3, f, "smooth") for f in range(1, DISTINCT)]
    B = max(FRAMES)
    xor = torch.arange(2 * B, dtype=torch.uint8, device=dev).view(-1, 1, 1, 1)
    frames = {}
    for l in labels:
        base = torch.from_numpy(np.stack([s[l] for s in host_sets])).to(dev)
        frames[l] = base[torch.arange(2 * B, device=dev) % DISTINCT] ^ xor
    batches = [{l: frames[l][b * B:(b + 1) * B] for l in labels} for b in range(2)]

    def launch(leg, b, F):
        L = legs[leg]
        L["plan"].run([batches[b][l][:F] for l in labels], out=L["out"][:F], n_frames=F)

    launch("seams", 0, 1)
    torch.cuda.synchronize()
    want = seam_model.blend_cv2(flat.layers, flat.out_w, flat.out_h, frames0, m, BANDS)
    frame0 = bool(np.array_equal(legs["seams"]["out"][0].cpu().numpy(), want))
    if not frame0:
        raise SystemExit("%s: frame 0 with seams differs from seam_model.blend_cv2" % name)
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
            res["F%d_%s" % (F, leg)] = dict(variant=variant[leg], ms_per_launch=[round(v, 4) for v in ms[leg]],
                                            ms_best=round(best, 4), panoramas_per_s=round(F / best * 1e3, 1))
    return dict(workload=name, cameras=n, frame_hw=[h, w], panorama_hw=[flat.out_h, flat.out_w], bands=BANDS,
                plan_time=plan_time, frame0_equals_cv2=frame0, launches_per_round=launches, rounds=rounds,
                per_frame=res)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", default="cfg2_6x1080p,ns_8x1080p")
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON record here")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_seams.py needs a CUDA device")
    torch.cuda.set_device(0)
    rec = dict(bench="seams", **gpu_info(torch),
               results=[run_workload(torch, w, args.launches, args.rounds, args.reps)
                        for w in args.workloads.split(",")])
    text = json.dumps(rec, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
