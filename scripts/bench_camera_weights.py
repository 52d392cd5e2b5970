"""Measurement of the camera-weighted blend (include/mcs.h mcs_plan_set_camera_weights) on one GPU.

Inputs resident in HBM, 64 frame-sets per launch, CUDA events around at least 100 timed launches
after a warm-up, two batches of distinct frame-sets alternated so that every launch reads inputs
(2.4 GB on config 2) far beyond the 126 MB of L2.  Per workload (config 2 = 6 x 1080p and
ns_8x1080p = 8 x 1080p, BGR) four legs, alternated round by round:
  ramp       edge ramps (``edge_ramp``, 64 px) on every camera: every overlap pixel is blended
  mask15     binary masks that blank the bottom 15 % of each camera: mostly one contributor a pixel
  overwrite  the reference's overwrite on the tiled kernel (variant 2)
  gather     the same overwrite forced onto the gather kernel (variant 1)
Before timing, frame 0 of each weighted leg is compared with the layer model of
oracle/camera_weight_model.py.  Reports ms per launch, panoramas/s, the algorithmic bytes
(out_w*out_h*C + C * sum of the contributions, mcs_plan_owned_pixels) and their rate as a fraction of
the HBM copy bandwidth, with the GPU name and power limit.

    python scripts/bench_camera_weights.py [--launches 100] [--rounds 3] [--out profiles/camera_weights.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {"cfg2_6x1080p": (6, 1080, 1920), "ns_8x1080p": (8, 1080, 1920)}
BATCH = 64
DISTINCT = 4   # host frame-sets; the device batches are XOR-ed copies of them, distinct per frame


def peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6533.5, "fallback (HBM copy bandwidth measured on a B200, BASELINE.md)"


def gpu_info(torch):
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [v.strip() for v in q.split(",")[:2]]
    except Exception as e:   # the record then says why the power limit is missing
        info["power_limit"] = "unknown (%s)" % e
    return info


def mask15(shape):
    m = np.full(shape[:2], 255, np.uint8)
    m[int(round(shape[0] * 0.85)):] = 0
    return m


def run_workload(torch, name, launches, rounds, check):
    from multicamera_stitching_b200 import edge_ramp, synthetic
    from multicamera_stitching_b200.plan import flatten_chain
    from oracle import camera_weight_model
    dev = torch.device("cuda", 0)
    n, h, w = WORKLOADS[name]
    st, _, labels, images = synthetic.synthetic_stitcher(n, h, w, 3, kind="smooth")
    shapes = [images[l].shape for l in labels]
    host_sets = [images] + [synthetic.make_frames(n, h, w, 3, f, "smooth") for f in range(1, DISTINCT)]
    # two batches of 2 * BATCH distinct frame-sets per camera: frame f = host set f % DISTINCT XOR f
    xor = torch.arange(2 * BATCH, dtype=torch.uint8, device=dev).view(-1, 1, 1, 1)
    frames = {}
    for l in labels:
        base = torch.from_numpy(np.stack([s[l] for s in host_sets])).to(dev)
        frames[l] = base[torch.arange(2 * BATCH, device=dev) % DISTINCT] ^ xor
    batches = [{l: frames[l][b * BATCH:(b + 1) * BATCH] for l in labels} for b in range(2)]

    legs = {}
    for leg, maps in (("ramp", {l: edge_ramp(images[l].shape, 64) for l in labels}),
                      ("mask15", {l: mask15(images[l].shape) for l in labels}), ("overwrite", None)):
        st.camera_weights = maps
        plan = st.plan(shapes, dev)
        out = plan.new_output(BATCH)
        legs[leg] = dict(plan=plan, out=out, maps=maps, force=0)
    legs["gather"] = dict(legs["overwrite"], force=1)
    st.camera_weights = None

    def launch(leg, b):
        L = legs[leg]
        L["plan"].handle.force_variant(L["force"])
        L["plan"].run([batches[b][l] for l in labels], out=L["out"], n_frames=BATCH)

    checks = {}
    for leg in ("ramp", "mask15"):
        launch(leg, 0)
        torch.cuda.synchronize()
        if check:
            flat = flatten_chain(st.stitchers, shapes)
            ref, _, _ = camera_weight_model.blend(flat.layers, flat.out_w, flat.out_h, [images[l] for l in labels],
                                                  [legs[leg]["maps"][l] for l in labels])
            checks[leg] = bool(np.array_equal(legs[leg]["out"][0].cpu().numpy(), ref))
            if not checks[leg]:
                raise SystemExit("%s %s: frame 0 differs from the layer model" % (name, leg))
    for leg in legs:   # warm-up of every leg and batch
        for b in (0, 1, 0, 1):
            launch(leg, b)
    torch.cuda.synchronize()

    ms = {leg: [] for leg in legs}
    variant = {}
    for _ in range(rounds):
        for leg in legs:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(launches):
                launch(leg, i & 1)
            e1.record()
            torch.cuda.synchronize()
            ms[leg].append(e0.elapsed_time(e1) / launches)
            variant[leg] = legs[leg]["plan"].handle.last_variant()
    peak, _ = peak_gbs()
    res = {}
    for leg in legs:
        plan = legs[leg]["plan"]
        plan.handle.force_variant(legs[leg]["force"])
        ab = plan.algorithmic_bytes() * BATCH
        best = min(ms[leg])
        res[leg] = dict(variant=variant[leg], ms_per_launch=[round(v, 4) for v in ms[leg]], ms_best=round(best, 4),
                        panoramas_per_s=round(BATCH / best * 1e3, 1), algorithmic_bytes_per_launch=int(ab),
                        achieved_gbs=round(ab / best / 1e6, 1), frac_of_hbm=round(ab / best / 1e6 / peak, 4))
        if leg in checks:
            res[leg]["frame0_equals_model"] = checks[leg]
    for leg in legs:
        legs[leg]["plan"].handle.force_variant(0)
    return dict(workload=name, cameras=n, frame_hw=[h, w], panorama_hw=[legs["ramp"]["plan"].out_h, legs["ramp"]["plan"].out_w],
                panoramas_per_launch=BATCH, launches_per_round=launches, rounds=rounds, legs=res)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", default="cfg2_6x1080p,ns_8x1080p")
    ap.add_argument("--launches", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--no-check", action="store_true", help="skip the comparison with the layer model")
    ap.add_argument("--out", default=None, help="also write the JSON record here")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_camera_weights.py needs a CUDA device")
    torch.cuda.set_device(0)
    peak, peak_src = peak_gbs()
    rec = dict(bench="camera_weights", **gpu_info(torch), hbm_gbs=peak, hbm_source=peak_src,
               results=[run_workload(torch, w, args.launches, args.rounds, not args.no_check)
                        for w in args.workloads.split(",")])
    text = json.dumps(rec, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
