"""Measurement of the exposure compensation of the camera-weighted and multi-band blends (include/mcs.h
mcs_plan_estimate_gains, mcs_plan_set_exposure_gains) on one GPU.

Per workload (config 2 = 6 x 1080p and ns_8x1080p = 8 x 1080p, BGR "smooth" synthetic frames, each camera at its own
brightness scale 0.7-1.3, edge ramps of 64 px as masks):
  estimation   mcs_plan_estimate_gains on frame-set 0 resident on the device (sample the weights and images, the
               statistics kernel, the solve), host clock around the synchronous call; against cv2's
               GainCompensator.feed on the same planes with 16 host threads (cv2.setNumThreads(16)).  The gains are
               compared: the statistics bit for bit with oracle/exposure_model.stats, the gains with its solve.
  per frame    variant 5 (camera-weighted blend) and variant 6 (multi-band blend, 5 bands) with the estimated gains and
               without, inputs resident in HBM, F = 16 panoramas per launch, legs alternated round by round, CUDA
               events.

    python scripts/bench_exposure.py [--launches 10] [--rounds 3] [--reps 3] [--out profiles/exposure.json]
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


def _scaled(frames, n):
    scale = np.random.default_rng(2).uniform(0.7, 1.3, n)
    return [np.clip(f.astype(np.float64) * s, 0, 255).astype(np.uint8) for f, s in zip(frames, scale)]


def run_workload(torch, name, launches, rounds, reps):
    import cv2
    from multicamera_stitching_b200 import _cabi, edge_ramp, synthetic
    from multicamera_stitching_b200.engine import CompiledPlan
    from multicamera_stitching_b200.plan import flatten_chain
    from oracle import exposure_model as ex
    from oracle import multiband_model as mb
    dev = torch.device("cuda", 0)
    n, h, w = WORKLOADS[name]
    st, _, labels, images = synthetic.synthetic_stitcher(n, h, w, 3, kind="smooth")
    shapes = [images[l].shape for l in labels]
    flat = flatten_chain(st.stitchers, shapes)
    frames0 = _scaled([images[l] for l in labels], n)
    m = [edge_ramp(f.shape, 64) for f in frames0]

    # estimation
    plan6 = CompiledPlan(flat, dev, camera_weights=m, blend_bands=BANDS)
    up = [torch.from_numpy(frames0[l.cam]).to(dev) for l in flat.layers]
    ptrs, pitches = [t.data_ptr() for t in up], [t.stride(0) for t in up]
    est = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        gains, N, I = plan6.handle.estimate_gains(ptrs, pitches, stats=True)
        est.append((time.perf_counter() - t0) * 1e3)
    planes = mb.camera_planes(flat.layers, flat.out_w, flat.out_h, frames0, m)
    inputs = ex.plane_inputs(planes)
    wN, wI, skip = ex.stats(*inputs)
    fed = plan6.handle.fed_layers()
    exact = bool(np.array_equal(N, wN) and np.array_equal(I, wI) and np.array_equal(gains[fed], ex.solve(wN, wI, skip)))
    if not exact:
        raise SystemExit("%s: the device statistics or gains differ from oracle/exposure_model" % name)
    cv2.setNumThreads(16)
    cv2_ms = []
    for _ in range(reps):
        t0 = time.perf_counter()
        want = ex.gains_cv2(*inputs)
        cv2_ms.append((time.perf_counter() - t0) * 1e3)
    largest = max(int(v) for i, row in enumerate(N) for j, v in enumerate(row) if i != j)
    estimation = dict(pairs=int(sum(1 for i in range(len(N)) for j in range(i + 1, len(N)) if N[i, j])),
                      largest_intersection_px=largest, device_ms=[round(v, 2) for v in est],
                      device_ms_best=round(min(est), 2), cpu_cv2_feed_ms=[round(v, 1) for v in cv2_ms],
                      cpu_cv2_feed_ms_best=round(min(cv2_ms), 1), stats_and_gains_equal_restatement=exact,
                      gains=[round(float(g), 6) for g in gains],
                      max_rel_diff_to_cv2=float(np.max(np.abs(gains[fed] - want) / np.abs(want))))
    del up

    # per frame: variants 5 and 6, with the gains and without
    legs = {}
    for variant, bands in ((5, 0), (6, BANDS)):
        for g in (None, gains):
            try:
                p = CompiledPlan(flat, dev, camera_weights=m, blend_bands=bands)
            except _cabi.McsError as e:   # more than 4 cameras on a pixel: the camera-weighted kernel refuses the rig
                legs["v%d" % variant] = str(e)
                break
            if g is not None:
                p.handle.set_exposure_gains(g)
            legs["v%d_%s" % (variant, "gains" if g is not None else "plain")] = p
    plans = {k: p for k, p in legs.items() if not isinstance(p, str)}
    outs = {leg: p.new_output(F) for leg, p in plans.items()}
    host_sets = [dict(zip(labels, frames0))] + [dict(zip(labels, _scaled([s[l] for l in labels], n)))
                                               for s in (synthetic.make_frames(n, h, w, 3, f, "smooth")
                                                         for f in range(1, DISTINCT))]
    xor = torch.arange(2 * F, dtype=torch.uint8, device=dev).view(-1, 1, 1, 1)
    frames = {}
    for l in labels:
        base = torch.from_numpy(np.stack([s[l] for s in host_sets])).to(dev)
        frames[l] = base[torch.arange(2 * F, device=dev) % DISTINCT] ^ xor
    batches = [{l: frames[l][b * F:(b + 1) * F] for l in labels} for b in range(2)]

    def launch(leg, b):
        plans[leg].run([batches[b][l] for l in labels], out=outs[leg], n_frames=F)

    for leg in plans:
        for b in (0, 1, 0, 1):
            launch(leg, b)
    torch.cuda.synchronize()
    ms = {leg: [] for leg in plans}
    for _ in range(rounds):
        for leg in plans:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(launches):
                launch(leg, i & 1)
            e1.record()
            torch.cuda.synchronize()
            ms[leg].append(e0.elapsed_time(e1) / launches)
    per_frame = {"F%d_%s" % (F, leg): dict(variant=plans[leg].handle.last_variant(),
                                           ms_per_launch=[round(v, 4) for v in ms[leg]], ms_best=round(min(ms[leg]), 4),
                                           panoramas_per_s=round(F / min(ms[leg]) * 1e3, 1)) for leg in plans}
    per_frame.update({k: v for k, v in legs.items() if isinstance(v, str)})
    return dict(workload=name, cameras=n, frame_hw=[h, w], panorama_hw=[flat.out_h, flat.out_w], bands=BANDS,
                estimation=estimation, launches_per_round=launches, rounds=rounds, per_frame=per_frame)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", default="cfg2_6x1080p,ns_8x1080p")
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON record here")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_exposure.py needs a CUDA device")
    torch.cuda.set_device(0)
    rec = dict(bench="exposure", **gpu_info(torch),
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
