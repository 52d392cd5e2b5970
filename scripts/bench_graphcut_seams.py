"""Measurement of the graph-cut seams of the multi-band blend (include/mcs.h mcs_plan_set_graphcut_seams) on one GPU.

Per workload (config 2 = 6 x 1080p and ns_8x1080p = 8 x 1080p, BGR "smooth" synthetic frames, edge ramps of 64 px
as masks, 5 bands; the seams are found on frame-set 0):
  plan time    mcs_plan_set_graphcut_seams(plan, frame-set) (sample the weights and images, one exact max flow per
               overlapping pair, rebuild the weight pyramids and sums) and (plan, NULL) (the rebuild alone), host
               clock around the synchronous call, alternated (on first, so that every off call rebuilds).  Per pair: the same call on a plan of the first two
               fed layers alone (the first pair of the full search, on the same masks).
  cv2          oracle/graphcut_seam_model.find_graphcut_cv2 (cv2's GraphCutSeamFinder("COST_COLOR")) on the planes of that
               first pair, once; cv2 runs one pair on one host thread, so the whole rig takes about the pair count
               times as long (not measured: minutes per workload).
  per frame    the multi-band blend with graph-cut seams and without, inputs resident in HBM, F = 16 panoramas per
               launch, legs alternated round by round, CUDA events.  Frame 0 of the seams leg is compared with
               oracle/graphcut_seam_model.blend_graphcut with --check (the device seams against the numpy restatement:
               scipy takes minutes per 1080-row pair, so it is off by default).

    python scripts/bench_graphcut_seams.py [--launches 10] [--rounds 3] [--reps 3] [--out profiles/graphcut_seams.json]
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
F = 16
BANDS = 5


def _timed(torch, fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


def run_workload(torch, name, launches, rounds, reps, check):
    from multicamera_stitching_b200 import edge_ramp, synthetic
    from multicamera_stitching_b200.engine import CompiledPlan
    from multicamera_stitching_b200.plan import FlatPlan, flatten_chain
    from oracle import multiband_model as mb
    from oracle import graphcut_seam_model, seam_model
    dev = torch.device("cuda", 0)
    n, h, w = WORKLOADS[name]
    st, _, labels, images = synthetic.synthetic_stitcher(n, h, w, 3, kind="smooth")
    shapes = [images[l].shape for l in labels]
    maps = {l: edge_ramp(images[l].shape, 64) for l in labels}
    flat = flatten_chain(st.stitchers, shapes)
    frames0, m = [images[l] for l in labels], [maps[l] for l in labels]
    planes = mb.camera_planes(flat.layers, flat.out_w, flat.out_h, frames0, m)
    sizes, corners, masks, imgs = graphcut_seam_model.plane_inputs(planes)
    pairs = seam_model.find(sizes, corners, [np.zeros_like(k) for k in masks], details=True)[1]
    st.camera_weights, st.blend_bands = maps, BANDS

    # plan time of the whole rig
    plan = CompiledPlan(flat, dev, camera_weights=m, blend_bands=BANDS)
    handle = plan.handle
    up = [torch.from_numpy(frames0[l.cam]).to(dev) for l in flat.layers]
    ptrs, pitches = [t.data_ptr() for t in up], [t.stride(0) for t in up]
    on, off = [], []
    for _ in range(reps):
        on.append(_timed(torch, lambda: handle.set_graphcut_seams(ptrs, pitches)))
        off.append(_timed(torch, lambda: handle.set_graphcut_seams(None, None)))
    handle.set_graphcut_seams(ptrs, pitches)
    assert handle.graphcut_seams

    # the first pair alone, on the device and in cv2
    fed = [l for l in flat.layers if min(flat.out_w, l.rect[2]) > max(0, l.rect[0])
           and min(flat.out_h, l.rect[3]) > max(0, l.rect[1])]
    two = FlatPlan(fed[:2], flat.out_w, flat.out_h, flat.channels, flat.ndim)
    pair_plan = CompiledPlan(two, dev, camera_weights=m, blend_bands=BANDS)
    up2 = [torch.from_numpy(frames0[l.cam]).to(dev) for l in two.layers]
    pair_ms = [_timed(torch, lambda: pair_plan.handle.set_graphcut_seams([t.data_ptr() for t in up2],
                                                                       [t.stride(0) for t in up2]))
               for _ in range(reps)]
    t0 = time.perf_counter()
    graphcut_seam_model.find_graphcut_cv2(sizes[:2], corners[:2], masks[:2], imgs[:2])
    cv2_pair_ms = (time.perf_counter() - t0) * 1e3
    roi = seam_model.overlap(sizes[0], corners[0], sizes[1], corners[1])
    plan_time = dict(pairs=len(pairs), largest_submask_wh=max(seam_model.submask_size(r) for _, _, r in pairs),
                     seams_on_ms=[round(v, 2) for v in on], seams_on_ms_best=round(min(on), 2),
                     rebuild_alone_ms=[round(v, 2) for v in off], rebuild_alone_ms_best=round(min(off), 2),
                     first_pair_submask_wh=seam_model.submask_size(roi),
                     first_pair_device_ms=[round(v, 2) for v in pair_ms], first_pair_device_ms_best=round(min(pair_ms), 2),
                     first_pair_cpu_cv2_ms=round(cv2_pair_ms, 1))
    del up, up2, pair_plan

    # per frame, with the seams and without
    legs = {"graphcut": plan, "no_seams": CompiledPlan(flat, dev, camera_weights=m, blend_bands=BANDS)}
    outs = {leg: p.new_output(F) for leg, p in legs.items()}
    host_sets = [images] + [synthetic.make_frames(n, h, w, 3, f, "smooth") for f in range(1, DISTINCT)]
    xor = torch.arange(2 * F, dtype=torch.uint8, device=dev).view(-1, 1, 1, 1)
    frames = {}
    for l in labels:
        base = torch.from_numpy(np.stack([s[l] for s in host_sets])).to(dev)
        frames[l] = base[torch.arange(2 * F, device=dev) % DISTINCT] ^ xor
    batches = [{l: frames[l][b * F:(b + 1) * F] for l in labels} for b in range(2)]

    def launch(leg, b):
        legs[leg].run([batches[b][l] for l in labels], out=outs[leg], n_frames=F)

    frame0 = None
    if check:
        launch("graphcut", 0)
        torch.cuda.synchronize()
        want = graphcut_seam_model.blend_graphcut(flat.layers, flat.out_w, flat.out_h, frames0, m, BANDS)
        frame0 = bool(np.array_equal(outs["graphcut"][0].cpu().numpy(), want))
        if not frame0:
            raise SystemExit("%s: frame 0 with graph-cut seams differs from graphcut_seam_model.blend_graphcut" % name)
    for leg in legs:
        for b in (0, 1, 0, 1):
            launch(leg, b)
    torch.cuda.synchronize()
    ms = {leg: [] for leg in legs}
    for _ in range(rounds):
        for leg in legs:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(launches):
                launch(leg, i & 1)
            e1.record()
            torch.cuda.synchronize()
            ms[leg].append(e0.elapsed_time(e1) / launches)
    per_frame = {"F%d_%s" % (F, leg): dict(variant=legs[leg].handle.last_variant(),
                                           ms_per_launch=[round(v, 4) for v in ms[leg]], ms_best=round(min(ms[leg]), 4),
                                           panoramas_per_s=round(F / min(ms[leg]) * 1e3, 1)) for leg in legs}
    return dict(workload=name, cameras=n, frame_hw=[h, w], panorama_hw=[flat.out_h, flat.out_w], bands=BANDS,
                plan_time=plan_time, frame0_equals_restatement=frame0, launches_per_round=launches, rounds=rounds,
                per_frame=per_frame)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", default="cfg2_6x1080p,ns_8x1080p")
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--check", action="store_true", help="compare frame 0 with the scipy restatement (slow)")
    ap.add_argument("--out", default=None, help="also write the JSON record here")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_graphcut_seams.py needs a CUDA device")
    torch.cuda.set_device(0)
    rec = dict(bench="graphcut_seams", **gpu_info(torch),
               results=[run_workload(torch, w, args.launches, args.rounds, args.reps, args.check)
                        for w in args.workloads.split(",")])
    text = json.dumps(rec, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
