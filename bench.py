#!/usr/bin/env python
"""Benchmark of the fused warp+paste compositing path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A *step* is one pass of the hot path over one batch of synthetic frame-sets.  Default workload: 8 x 1080p
cameras into one panorama - the geometry north_star's 70 % target is quoted on - with 5 launches of 64
frame-sets per step (20 steps time 100 launches; inputs 3.2 GB + outputs 2.1 GB per launch, far beyond the
126 MB L2, so no launch sees a warm cache).  BASELINE.json's other configurations ride along as ``extra``
records of the same line: config 2 (6 x 1080p) and config 3 (8 x 2160p) device-resident with their roofline
fractions, config 4 (recalibration of four 1080p pairs through the batched matchKeypoints, host refit
included) and config 5 (a 10 000-frame 6 x 1080p sequence sharded by frame range, end to end).
Rank 0 prints ONE JSON line:

  value     panoramas/s, whole job, inputs already resident in HBM
  e2e       the same metric through the host-facing sequence API: pinned host
            frames -> H2D -> kernel -> D2H -> pinned host panoramas, every step
  roofline  algorithmic bytes per launch / CUDA-event launch duration against
            the measured HBM copy bandwidth (MEASURED_PEAKS.json)
  cpu_baseline  the reference's own OpenCV chain (oracle/stitcher_ref.py) timed
            on this box's host cores on a bounded sample of the same workload

``--impl reference`` times only that CPU chain (all host threads) and prints
the same line shape with ``"impl": "reference"``.

``--dump-outputs DIR`` (rank 0) writes what the timed paths computed in their last step, for comparing two builds
output for output (the synthetic inputs are seeded, so the same arguments give the same inputs):
``panoramas.npy`` from the timed launches (or the CPU chain with ``--impl reference``) and ``e2e_panoramas.npy``
from the end-to-end leg.  Each is a seeded sample of pixels, ``[K, C]`` float32, with their (frame, row, column)
in ``<name>_pixels.npy``, ``[K, 3]`` float32.

With N > 1 (torchrun, one rank per GPU) the sequence shards by frame range:
every rank composites its own batch, there is no data-path collective
(torch.distributed is used for the barrier and the max-over-ranks time only).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (n_cams, H, W, frame-sets per launch, e2e frame-sets per step)
    "cfg1_3x720p": (3, 720, 1280, 64, 64),
    "cfg2_6x1080p": (6, 1080, 1920, 64, 32),
    "cfg3_8x2160p": (8, 2160, 3840, 64, 8),
    "ns_8x1080p": (8, 1080, 1920, 64, 32),     # the geometry north_star's 70 % target names
}
DEFAULT_WORKLOAD = "ns_8x1080p"
LAUNCHES_PER_STEP = 5
FALLBACK_HBM_GBS = 6650.0
DUMP_PIXELS = 1 << 20   # pixels sampled per dumped output: 2 x 12 MB with their positions, two outputs < 64 MB


def build_chain(name):
    """Calibrated Stitcher of a workload plus what the CPU legs need: ``(stitcher, stage homographies, labels,
    images_dic)`` (host only; nothing of the oracle is touched here)."""
    from multicamera_stitching_b200 import synthetic
    n, h, w, _, _ = WORKLOADS[name]
    return synthetic.synthetic_stitcher(n, h, w, 3, kind="smooth")


def oracle_states(homographies, labels, images):
    """The CPU checker's states for the same chain (parity spot-check and CPU baseline legs only)."""
    from oracle import stitcher_ref
    return stitcher_ref.calibrate_chain_from_homographies([images[l].shape for l in labels], homographies)


def recorded_traffic(workload, batch):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture (None if the
    capture was taken at another batch size or does not exist)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_dram_traffic.json")) as f:
            rec = json.load(f)[workload]
        if int(rec["panoramas_per_launch"]) != int(batch):
            return None
        return int(rec["dram_read_bytes"]) + int(rec["dram_write_bytes"])
    except Exception:
        return None


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


def dump_outputs(out_dir, name, panos, seed=0):
    """Writes a fixed, seeded sample of the pixels of ``panos`` ([F, H, W(, C)] uint8, numpy or torch on any device)
    as ``out_dir/<name>.npy`` and their (frame, row, column) as ``out_dir/<name>_pixels.npy``, both float32."""
    shape = tuple(int(v) for v in panos.shape[:3])
    n = int(np.prod(shape))
    flat = np.arange(n) if n <= DUMP_PIXELS else np.unique(np.random.default_rng(seed).integers(0, n, DUMP_PIXELS))
    f, y, x = np.unravel_index(flat, shape)
    if isinstance(panos, np.ndarray):
        vals = panos[f, y, x]
    else:
        import torch
        f_t, y_t, x_t = (torch.from_numpy(a).to(panos.device) for a in (f, y, x))
        vals = panos[f_t, y_t, x_t].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), vals.astype(np.float32))
    np.save(os.path.join(out_dir, name + "_pixels.npy"), np.stack([f, y, x], axis=1).astype(np.float32))


# ---------------------------------------------------------------------------
class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                parts = [p.strip() for p in line.split(",")]
                if len(parts) < 7:
                    continue
                try:
                    sm.append(float(parts[0]))
                    mx.append(float(parts[1]))
                except ValueError:
                    continue
                for nm, v in zip(names, parts[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            os.unlink(self.path)
        except Exception:
            pass
        self.sm, self.mx, self.reasons = sm, mx, reasons
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out

    @staticmethod
    def merged(*samplers):
        """One clocks record over the timed regions of several samplers."""
        sm, mx, reasons = [], [], set()
        for s in samplers:
            sm += getattr(s, "sm", [])
            mx += getattr(s, "mx", [])
            reasons |= getattr(s, "reasons", set())
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": sorted(reasons), "samples": len(sm)}
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx))
        return out


# ---------------------------------------------------------------------------
def cpu_chain_runner(states, labels, images, homographies):
    """``(run(frame_set) -> panorama, kind, description)`` of the CPU arm: the reference's own ``Stitcher`` class where
    oracle/_ref exists (``kind`` "reference"), else the cv2 restatement of its chain (``kind`` "port")."""
    import cv2
    from oracle import build_ref, stitcher_ref
    ref_mod = None if os.environ.get("MCS_BENCH_REFERENCE_PORT") else build_ref.load()
    if ref_mod is not None:
        rs = build_ref.calibrated_stitcher(ref_mod, images, homographies)
        return (lambda fs: rs.stitch(fs)), "reference", (
            "the reference's own Stitcher.stitch (StitcherClass.py:114-136 through oracle/_ref, built by "
            "oracle/build_ref.py), cv2 %s" % cv2.__version__)
    return (lambda fs: stitcher_ref.stitch_chain(states, labels, fs)), "port", (
        "cv2 %s chain (warpPerspective + paste, StitcherClass.py:131-136, :239-241; oracle/stitcher_ref.py, pinned "
        "against the reference's own StitcherClass.py by tests/test_oracle_ref_pin.py)" % cv2.__version__)


def time_cpu_chain(run, frame_sets, budget_s, min_panos=4, threads=None):
    """Reference CPU path: the sequential cv2 chain of StitcherClass.py:131-136 (``run`` from cpu_chain_runner)."""
    import cv2
    if threads is not None:
        cv2.setNumThreads(threads)
    for fs in frame_sets[:2]:
        run(fs)  # warm-up
    n = 0
    t0 = time.perf_counter()
    while True:
        run(frame_sets[n % len(frame_sets)])
        n += 1
        dt = time.perf_counter() - t0
        if (dt >= budget_s and n >= min_panos) or n >= 100000:
            break
    return n / dt, n, dt, cv2.getNumThreads()


def make_frame_sets_offset(name, count, first_frame):
    from multicamera_stitching_b200 import synthetic
    n, h, w, _, _ = WORKLOADS[name]
    return [synthetic.make_frames(n, h, w, 3, frame_index=first_frame + f, kind="smooth") for f in range(count)]


# ---------------------------------------------------------------------------
def run_reference(args, rank, world):
    """The reference arm: the reference's OWN ``Stitcher`` class (PostScripts/Stitcher/StitcherClass.py, made
    importable by oracle/build_ref.py -> oracle/_ref, a build output that travels to the GPU box) calibrated with the
    workload's stage homographies and timed through its own ``stitch(images_dic)`` on all host threads.  Where
    that build output is missing, the cv2 restatement of the same chain (oracle/stitcher_ref.py) is timed."""
    if rank != 0:
        return
    st, homographies, labels, images = build_chain(args.workload)
    frame_sets = make_frame_sets_offset(args.workload, 4, 0)
    import cv2
    from oracle import stitcher_ref
    cv2.setNumThreads(os.cpu_count() or 1)
    states = oracle_states(homographies, labels, images)
    check = stitcher_ref.stitch_chain(states, labels, frame_sets[0])
    run, kind, what = cpu_chain_runner(states, labels, images, homographies)
    ref = run(frame_sets[0])
    if not np.array_equal(ref, check):
        raise SystemExit("bench.py: the reference arm and its restatement disagree")
    out_h, out_w = ref.shape[:2]
    per_step = args.ref_panos_per_step
    for _ in range(args.warmup):
        for i in range(per_step):
            run(frame_sets[i % 4])
    last = []
    t0 = time.perf_counter()
    for step in range(args.steps):
        for i in range(per_step):
            pano = run(frame_sets[i % 4])
            if args.dump_outputs and step == args.steps - 1:
                last.append(pano)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "panoramas", np.stack(last))
    pps = args.steps * per_step / dt
    line = {
        "impl": "reference", "metric": "panoramas_per_sec", "value": pps, "unit": "panoramas/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "output_mp_per_s": pps * out_w * out_h / 1e6,
        "config": {"workload": args.workload, "cameras": WORKLOADS[args.workload][0],
                   "frame_hw": list(WORKLOADS[args.workload][1:3]), "panorama_wh": [out_w, out_h],
                   "panoramas_per_step": per_step},
        "cpu_baseline": {"value": pps, "unit": "panoramas/s", "cores": cv2.getNumThreads(), "kind": kind,
                         "sample": "%d steps x %d panoramas, %s, %d threads"
                                   % (args.steps, per_step, what, cv2.getNumThreads())},
        "e2e": {"value": pps, "unit": "panoramas/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------
class Resident(object):
    """One workload resident in HBM: calibrated stitcher, compiled plan, a batch of frame-sets, the output batch."""

    def __init__(self, name, device, rank, batch=0, feather=0, pitch_align=128):
        import torch
        self.name = name
        n_cams, H, W, b, e2e_b = WORKLOADS[name]
        self.batch = batch or b
        self.e2e_batch = batch or e2e_b
        self.st, self.homographies, self.labels, self.images = build_chain(name)
        self.st.feather_log2 = feather   # 0 = the reference's overwrite (the headline); n = feather over 2**n px
        self.shapes = [self.images[l].shape for l in self.labels]
        self.plan = self.st.plan(self.shapes, device)
        self.algo_bytes = self.plan.algorithmic_bytes()
        # device-resident ring of distinct frame-sets (cycled to fill the batch); rank r starts at frame r * batch
        self.distinct = min(self.batch, 8 if H < 2000 else 4)
        self.ring = make_frame_sets_offset(name, self.distinct, rank * self.batch)
        self.dev_frames = {}
        for l in self.labels:
            stack = np.stack([self.ring[f % self.distinct][l] for f in range(self.batch)])
            self.dev_frames[l] = torch.from_numpy(stack).to(device)
        # panorama rows padded to a 128-byte pitch in HBM: every 128-column cell row of the tiled kernel then
        # starts and ends on a 32-byte sector boundary (no partial-sector writes)
        self.out = self.plan.new_output(self.batch, pitch_align=pitch_align)
        self.in_bytes = sum(int(t.numel()) for t in self.dev_frames.values())

    def launch(self):
        self.st.stitch_batch(self.dev_frames, out=self.out)

    def parity(self, feather=0):
        """GPU panorama 0 against the CPU chain (outside every timed region)."""
        import torch
        from oracle import stitcher_ref
        states = oracle_states(self.homographies, self.labels, self.images)
        self.launch()
        torch.cuda.synchronize()
        if feather:
            from oracle import feather_model
            ref = feather_model.feather_chain(states, self.labels, self.ring[0], feather)
        else:
            ref = stitcher_ref.stitch_chain(states, self.labels, self.ring[0])
        got = self.out[0].cpu().numpy()
        d = np.abs(got.astype(np.int16) - ref.astype(np.int16))
        return {"max_abs_diff": int(d.max()), "exact_fraction": float((d == 0).mean())}, ref, states

    def free(self):
        import torch
        self.dev_frames = self.out = self.plan = None
        torch.cuda.empty_cache()


def time_resident(w, ctx, steps, warmup, launches_per_step, sampler=None, clear_out=False):
    """CUDA-event time of ``steps`` steps of ``launches_per_step`` launches, max over ranks.  ``clear_out`` zeroes the
    output after the warm-up (untimed), so that what it holds afterwards was written by the timed launches."""
    import torch
    from multicamera_stitching_b200 import _cabi
    for _ in range(warmup):
        for _ in range(launches_per_step):
            w.launch()
    if clear_out:
        w.out.zero_()
    ctx.barrier()
    if sampler is not None:
        sampler.start()
    launches0 = _cabi.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        for _ in range(launches_per_step):
            w.launch()
    e1.record()
    ctx.barrier()
    launches = _cabi.launch_count() - launches0
    return ctx.max_over_ranks(e0.elapsed_time(e1)), launches


def host_ceiling(ctx, device, seconds=0.25):
    """What the box's host<->device path delivers when EVERY rank copies at once with nothing else going on:
    plain pinned 256 MB cudaMemcpyAsync in both directions on two streams, summed over the ranks (GB/s)."""
    import torch
    n = 256 << 20
    h_in, h_out = torch.empty(n, dtype=torch.uint8, pin_memory=True), torch.empty(n, dtype=torch.uint8, pin_memory=True)
    d_in, d_out = torch.empty(n, dtype=torch.uint8, device=device), torch.empty(n, dtype=torch.uint8, device=device)
    s_up, s_dn = torch.cuda.Stream(), torch.cuda.Stream()
    reps = 1
    for trial in range(2):   # first a probe for the repetition count, then the measurement
        ctx.barrier()
        e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        e[0].record(s_up)
        e[2].record(s_dn)
        for _ in range(reps):
            with torch.cuda.stream(s_up):
                d_in.copy_(h_in, non_blocking=True)
            with torch.cuda.stream(s_dn):
                h_out.copy_(d_out, non_blocking=True)
        e[1].record(s_up)
        e[3].record(s_dn)
        torch.cuda.synchronize()
        ms_up, ms_dn = e[0].elapsed_time(e[1]), e[2].elapsed_time(e[3])
        if trial == 0:
            reps = max(2, int(seconds * 1e3 / max(ms_up, ms_dn, 1e-3)))
    up = ctx.sum_over_ranks(n * reps / ms_up / 1e6)
    dn = ctx.sum_over_ranks(n * reps / ms_dn / 1e6)
    return up, dn


def extra_resident(name, device, rank, ctx, world, peak, steps=4, launches=3):
    """Another BASELINE configuration device-resident: panoramas/s, roofline fraction, parity of panorama 0."""
    w = Resident(name, device, rank)
    parity, _, _ = w.parity() if rank == 0 else (None, None, None)
    ms, n_launch = time_resident(w, ctx, steps, 3, launches)
    pps = world * w.batch * steps * launches / (ms * 1e-3)
    achieved = w.algo_bytes * w.batch * steps * launches / (ms * 1e-3) / 1e9
    rec = {"workload": name, "value": pps, "unit": "panoramas/s", "panoramas_per_launch": w.batch, "launches": n_launch,
           "launch_ms": ms / max(n_launch, 1), "output_mp_per_s": pps * w.plan.out_w * w.plan.out_h / 1e6,
           "panorama_wh": [w.plan.out_w, w.plan.out_h], "algorithmic_bytes_per_panorama": w.algo_bytes,
           "roofline_frac": achieved / peak, "achieved_gbs": achieved, "parity": parity}
    w.free()
    return rec


def extra_recalibration(device, budget_s=4.0):
    """BASELINE config 4 through the product's batched ``matchKeypoints``: ORB-2000 descriptors of four synthetic
    1080p pairs (detected on the host, outside the timed region, SURVEY section 8 a6), then per call ONE Hamming
    matching launch + ONE RANSAC scoring launch over the four pairs, uploads, downloads and the host refit
    included.  The cv2 arm runs the same four pairs through BFMatcher.knnMatch + the ratio loop +
    findHomography(RANSAC) on all host threads."""
    import cv2
    import torch
    from multicamera_stitching_b200 import StitcherBase, recalib, synthetic
    from oracle import stitcher_ref
    items = []
    for k in range(4):
        imageB, imageA, _ = synthetic.make_pair(1080, 1920, seed=k)
        sb = StitcherBase()
        kA, fA = sb.detectAndDescribe(imageA)
        kB, fB = sb.detectAndDescribe(imageB)
        items.append((kA, kB, fA, fB))
    res = recalib.match_keypoints_batch(items, 0.75, 3.0)      # warm-up, also the parity sample
    torch.cuda.synchronize()
    exact = True
    for item, (H, matches, status) in zip(items, res):
        Hc, mc, sc = stitcher_ref.match_keypoints(*item, ratio=0.75, reprojThresh=3.0)
        exact = exact and matches == mc
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < budget_s / 2 or n < 3:
        recalib.match_keypoints_batch(items, 0.75, 3.0)
        n += 1
    torch.cuda.synchronize()
    gpu = 4 * n / (time.perf_counter() - t0)
    # the matching kernel alone, descriptors resident (north_star: "the matcher reports INT/popcount pipe utilisation")
    nq_max, nt_max = max(len(i[2]) for i in items), max(len(i[3]) for i in items)
    dq = torch.zeros((4, nq_max, 32), dtype=torch.uint8, device=device)
    dt_ = torch.zeros((4, nt_max, 32), dtype=torch.uint8, device=device)
    for j, (_, _, fa, fb) in enumerate(items):
        dq[j, :len(fa)] = torch.from_numpy(np.ascontiguousarray(fa)).to(device)
        dt_[j, :len(fb)] = torch.from_numpy(np.ascontiguousarray(fb)).to(device)
    for _ in range(5):
        recalib.match_top2_batch(dq, dt_, ratio=0.75)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(50):
        recalib.match_top2_batch(dq, dt_, ratio=0.75)
    e1.record()
    torch.cuda.synchronize()
    match_ms = e0.elapsed_time(e1) / 50
    popc = 4 * nq_max * nt_max * 8      # 32-bit popcounts per launch (SURVEY section 8 d)
    cv2.setNumThreads(os.cpu_count() or 1)
    m, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < budget_s / 2 or m < 2:
        for item in items:
            stitcher_ref.match_keypoints(*item, ratio=0.75, reprojThresh=3.0)
        m += 1
    cpu = 4 * m / (time.perf_counter() - t0)
    return {"workload": "cfg4: 4 x 1080p pairs, ORB-2000, Hamming 2-NN + ratio test + RANSAC homography",
            "value": gpu, "unit": "pairs/s", "api": "recalib.match_keypoints_batch (StitcherBase.matchKeypoints for 4 pairs: "
            "1 matching + 1 RANSAC launch, host refit included, numpy in / numpy out)",
            "keypoints": [int(len(i[2])) for i in items], "match_lists_equal_cv2": bool(exact),
            "match_kernel": {"ms_per_launch": match_ms, "popc32_per_s": popc / (match_ms * 1e-3),
                             "xu_popc_pipe_pct_of_peak": 68.6, "alu_pipe_pct_of_peak": 36.0, "tensor_pipe_pct": 0.0,
                             "pipe_source": "ncu --set full, profiles/r1_match_ncu_full.txt (the kernel is unchanged since)"},
            "cpu_pairs_per_s": cpu, "cpu_threads": cv2.getNumThreads(), "n_gpus_used": 1}


def extra_sequence(device, rank, world, ctx, frames, chunk):
    """BASELINE config 5: a ``frames``-frame 6 x 1080p sequence sharded by frame range, pinned host frames in,
    pinned host panoramas out, through ``SequencePipeline.run(ring=True)`` (a ring of 32 frame-sets per rank)."""
    import torch
    from multicamera_stitching_b200 import synthetic
    from multicamera_stitching_b200.sequence import SequencePipeline, pinned_like, shard_range
    st, homographies, labels, images = build_chain("cfg2_6x1080p")
    shapes = [images[l].shape for l in labels]
    pipe = SequencePipeline(st, shapes, device, chunk=chunk, depth=3)
    R, distinct = 32, 8
    sets = [synthetic.make_frames(6, 1080, 1920, 3, frame_index=rank * 1000 + f, kind="smooth") for f in range(distinct)]
    host = {l: pinned_like((R,) + tuple(images[l].shape)) for l in labels}
    for l in labels:
        for f in range(R):
            host[l][f].copy_(torch.from_numpy(sets[f % distinct][l]))
    out = pinned_like((R,) + pipe.plan.out_shape())
    lo, hi = shard_range(frames, world, rank)
    pipe.run(host, out, lo, min(hi, lo + 2 * R), ring=True)
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    pipe.run(host, out, lo, hi, ring=True)
    e1.record()
    ctx.barrier()
    ms = ctx.max_over_ranks(e0.elapsed_time(e1))
    h2d, d2h = pipe.bytes_per_frame()
    del pipe, host, out
    torch.cuda.empty_cache()
    return {"workload": "cfg5: %d-frame 6 x 1080p sequence, frame-range shards, end to end" % frames,
            "value": frames / (ms * 1e-3), "unit": "panoramas/s", "seconds": ms * 1e-3,
            "h2d_bytes_per_panorama": h2d, "d2h_bytes_per_panorama": d2h,
            "host_to_device_gbs": h2d * frames / ms / 1e6, "device_to_host_gbs": d2h * frames / ms / 1e6,
            "collectives_on_data_path": 0}


def extra_blend(device, rank, world, ctx, peak, feather=3, chunk=16):
    """BASELINE config 2's "feather blend" on its own geometry (6 x 1080p): every paste softened over 2**feather
    pixels, the seam bands blended inside the tiled kernel (BAND tiles, one launch).  Device-resident rate and
    parity against the blend specification (oracle/feather_model.py; ours - the reference only overwrites), and
    the end-to-end rate through the sequence pipeline, which keeps its window uploads in this mode."""
    import torch
    from multicamera_stitching_b200.sequence import SequencePipeline, pinned_like
    w = Resident("cfg2_6x1080p", device, rank, feather=feather)
    parity, _, _ = w.parity(feather) if rank == 0 else (None, None, None)
    ms, n_launch = time_resident(w, ctx, 4, 3, 3)
    pps = world * w.batch * 4 * 3 / (ms * 1e-3)
    stats = w.plan.handle.tiled_stats()
    variant = w.plan.handle.last_variant()
    pipe = SequencePipeline(w.st, w.shapes, device, chunk=chunk, depth=3)
    R = 32
    host = {l: pinned_like((R,) + tuple(w.images[l].shape)) for l in w.labels}
    for l in w.labels:
        for f in range(R):
            host[l][f].copy_(torch.from_numpy(w.ring[f % w.distinct][l]))
    out = pinned_like((R,) + w.plan.out_shape())
    pipe.run(host, out)
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    pipe.run(host, out, 0, 8 * R, ring=True)
    e1.record()
    ctx.barrier()
    e2e_ms = ctx.max_over_ranks(e0.elapsed_time(e1))
    h2d, d2h = pipe.bytes_per_frame()
    whole = sum(int(np.prod(sh)) for sh in w.shapes)
    del pipe, host, out
    w.free()
    torch.cuda.empty_cache()
    return {"workload": "cfg2 geometry, feather blend over %d px (reference: overwrite only)" % (1 << feather),
            "value": pps, "unit": "panoramas/s", "launch_ms": ms / max(n_launch, 1), "kernel_variant": variant,
            "band_tiles": stats.get("band"), "band_fused": stats.get("band_fused"), "tiles": stats.get("tiles"),
            "parity_vs_blend_specification": parity,
            "e2e_panoramas_per_s": world * 8 * R / (e2e_ms * 1e-3), "h2d_bytes_per_panorama": h2d,
            "whole_frame_bytes_per_panorama": whole, "d2h_bytes_per_panorama": d2h}


def extra_recorded(device, n_sets=48, quality=90):
    """A recorded capture in the reference's own format (data.csv + JPEG files, data_capture_node.py:107-130) on
    config 2's geometry, composited through ``recorded.stitch_capture``: JPEG decode on the host thread pool one
    batch ahead of the pipeline (video_mapping_node.py:105-130 replays while it stitches).  Rank 0 only."""
    import shutil
    import torch
    from multicamera_stitching_b200 import recorded, synthetic
    st, homographies, labels, images = build_chain("cfg2_6x1080p")
    tmp = tempfile.mkdtemp(prefix="mcs_capture_")
    try:
        distinct = [synthetic.make_frames(6, 1080, 1920, 3, frame_index=f, kind="smooth") for f in range(4)]
        recorded.write_capture(tmp, [distinct[f % 4] for f in range(n_sets)], quality=quality)
        seq = recorded.RecordedSequence(tmp)
        runner = recorded.CaptureRunner(st, seq, device=device, batch=16)     # pipeline + pinned buffers, once
        out = torch.empty((n_sets,) + runner.out_shape(), dtype=torch.uint8, pin_memory=True)
        runner.run(0, 32, out[:32])                                           # warm-up (plan, page cache)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        panos = runner.run(0, n_sets, out)
        dt = time.perf_counter() - t0
        t1 = time.perf_counter()
        runner._decode(0, 0, 16)            # the JPEG decode alone, into the runner's pinned buffers
        decode = 16 / (time.perf_counter() - t1)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return {"workload": "recorded capture: %d frame-sets of 6 x 1080p JPEG (quality %d), data.csv format of the reference"
                        % (n_sets, quality),
            "value": n_sets / dt, "unit": "panoramas/s", "api": "recorded.CaptureRunner.run (decode-ahead, SequencePipeline; buffers allocated once)",
            "decode_only_frame_sets_per_s": decode, "decode_threads": min(16, os.cpu_count() or 1),
            "panoramas": int(panos.shape[0])}


def extra_single_call(device, calls=20):
    """The reference's own call shape, one frame-set per call: ``Stitcher.stitch(images_dic)`` with numpy frames in
    (pageable host memory) and a numpy panorama of its own out (StitcherClass.py:114-136), on config 2, next to the
    cv2 chain on all host threads with the same frames.  Rank 0 only; wall clock, every call blocking."""
    import cv2
    import torch
    from oracle import stitcher_ref
    st, homographies, labels, images = build_chain("cfg2_6x1080p")
    states = oracle_states(homographies, labels, images)
    with torch.cuda.device(device):
        got = st.stitch(images)
        ref = stitcher_ref.stitch_chain(states, labels, images)
        st.stitch(images)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(calls):
            st.stitch(images)
        ms = (time.perf_counter() - t0) / calls * 1e3
    cv2.setNumThreads(os.cpu_count() or 1)
    t0 = time.perf_counter()
    for _ in range(4):
        stitcher_ref.stitch_chain(states, labels, images)
    ms_cv2 = (time.perf_counter() - t0) / 4 * 1e3
    return {"workload": "cfg2_6x1080p, one frame-set per call", "api": "Stitcher.stitch(images_dic): numpy frames in, numpy panorama out",
            "ms_per_call": ms, "value": 1e3 / ms, "unit": "panoramas/s", "bit_exact_vs_cv2": bool(np.array_equal(got, ref)),
            "cv2_chain_ms_per_call": ms_cv2, "cv2_threads": os.cpu_count() or 1,
            "h2d_bytes_per_call": int(sum(w["nbytes"] * w["rows"] for b in st._engine_().plan_for(
                st.stitchers, [images[l].shape for l in labels], device).upload_bands().values() for w in b[2])),
            "d2h_bytes_per_call": int(got.nbytes)}


# ---------------------------------------------------------------------------
def run_ours(args, rank, local_rank, world):
    import torch
    from multicamera_stitching_b200 import _cabi
    from multicamera_stitching_b200.sequence import SequencePipeline, pinned_like
    from multicamera_stitching_b200.shard import ShardContext, bind_to_gpu_numa

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback for the GPU arm)")
    _cabi.load()
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    # pinned buffers of this rank on its GPU's socket ($MCS_BENCH_NO_NUMA=1 leaves the threads alone)
    numa_bound = False if os.environ.get("MCS_BENCH_NO_NUMA") else bind_to_gpu_numa(local_rank)
    # control path only (barrier, max / sum of scalars): gloo on the host, the GPUs never talk to each other
    ctx = ShardContext.from_env(backend="gloo", device=None)
    _barrier = ctx.barrier

    def barrier():
        torch.cuda.synchronize()
        _barrier()
    ctx.barrier = barrier
    max_over_ranks = ctx.max_over_ranks

    w = Resident(args.workload, device, rank, batch=args.batch, feather=args.feather, pitch_align=args.pitch_align)
    n_cams, H, W = WORKLOADS[args.workload][:3]
    batch, e2e_batch = w.batch, w.e2e_batch
    out_w, out_h = w.plan.out_w, w.plan.out_h
    parity, ref, states = w.parity(args.feather) if rank == 0 else (None, None, None)
    if rank == 0 and (parity["max_abs_diff"] > 1 or parity["exact_fraction"] < 0.999) and not os.environ.get("MCS_BENCH_ABLATION"):
        raise SystemExit("bench.py: GPU panorama differs from the cv2 chain: %r" % (parity,))

    # ---- kernel-resident timing ------------------------------------------------
    lps = args.launches_per_step
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ms_total, launches = time_resident(w, ctx, args.steps, args.warmup, lps, sampler, clear_out=bool(args.dump_outputs))
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, "panoramas", w.out)   # every launch of the last step wrote w.out
    ms_step = ms_total / args.steps
    pps = world * batch * lps * args.steps / (ms_total * 1e-3)
    launch_ms = ms_total / max(launches, 1)
    kernels_per_launch_call = launches / max(args.steps * lps, 1)   # 1 in overwrite mode, 2 with the feather band pass
    # algorithmic bytes of one stitch call over its time (the feather mode adds a second, small launch over the seam bands)
    achieved = w.algo_bytes * batch * lps / (ms_step * 1e-3) / 1e9
    peak, peak_src = measured_peak()
    stats = w.plan.handle.tiled_stats()
    variant = w.plan.handle.last_variant()
    ctas = w.plan.handle.tiled_ctas_per_sm()

    if args.no_e2e:   # kernel experiments only: the line then carries no end-to-end number
        ctx.close()
        if rank == 0:
            print(json.dumps({"metric": "panoramas_per_sec", "value": pps, "ms_per_step": ms_step, "launch_ms": launch_ms,
                              "roofline": {"achieved": achieved, "frac": achieved / peak}, "parity": parity,
                              "gpu_launches": launches, "clocks": clocks, "e2e": None,
                              "ctas_per_sm": ctas, "tiled": stats}), flush=True)
        return

    # ---- end to end through the host-facing sequence API -------------------------
    pipe = SequencePipeline(w.st, w.shapes, device, chunk=args.chunk, depth=3, windows=not args.whole_frames)
    host_frames = {l: pinned_like((e2e_batch,) + tuple(w.images[l].shape)) for l in w.labels}
    for l in w.labels:
        for f in range(e2e_batch):
            host_frames[l][f].copy_(torch.from_numpy(w.ring[f % w.distinct][l]))
    host_out = pinned_like((e2e_batch,) + w.plan.out_shape())
    h2d_b, d2h_b = pipe.bytes_per_frame()
    for _ in range(max(1, min(args.warmup, 3))):
        pipe.run(host_frames, host_out)
    barrier()
    if rank == 0:
        got = host_out[0].numpy()
        d = np.abs(got.astype(np.int16) - ref.astype(np.int16))
        if int(d.max()) > 1:
            raise SystemExit("bench.py: e2e panorama differs from the cv2 chain")
    e2e_steps = args.steps
    if args.dump_outputs:
        host_out.zero_()   # untimed: the dump must come from the timed steps, not from the warm-up
    sampler2 = ClockSampler(local_rank)
    if rank == 0:
        sampler2.start()
    # The steps are consecutive batches of one streaming pipeline: frame f of the timed sequence lives
    # in slot f % batch of the pinned input ring and its panorama lands in the same slot of the pinned
    # output ring, so every step uploads its inputs and downloads its panoramas, and the pipeline is
    # not drained between steps (it is at the end: run() returns after the last device->host copy).
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    pipe.run(host_frames, host_out, 0, e2e_steps * e2e_batch, ring=True)
    e1.record()
    barrier()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1))
    if rank == 0:
        sampler2.stop()
        clocks = ClockSampler.merged(sampler, sampler2)   # both timed regions
    e2e_pps = world * e2e_batch * e2e_steps / (e2e_ms * 1e-3)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, "e2e_panoramas", host_out)   # the last step filled every slot of the ring
    del pipe, host_frames, host_out
    # what the box's host<->device path can carry with all ranks copying at once, and the panorama rate it allows
    up_gbs, dn_gbs = host_ceiling(ctx, device)
    ceiling_pps = min(up_gbs * 1e9 / max(h2d_b, 1), dn_gbs * 1e9 / max(d2h_b, 1))

    # ---- CPU baseline (rank 0, N = 1 only): the reference's cv2 chain ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        import cv2
        run_cpu, kind, what = cpu_chain_runner(states, w.labels, w.images, w.homographies)
        if not np.array_equal(run_cpu(w.ring[0]), ref):
            raise SystemExit("bench.py: the CPU arm and its restatement disagree")
        cpu_pps, n, dt, threads = time_cpu_chain(run_cpu, w.ring[:4], args.cpu_budget * 0.75, threads=os.cpu_count() or 1)
        one_pps, _, _, _ = time_cpu_chain(run_cpu, w.ring[:4], args.cpu_budget * 0.25, min_panos=2, threads=1)
        cpu = {"value": cpu_pps, "unit": "panoramas/s", "cores": threads, "single_thread_value": one_pps, "kind": kind,
               "sample": "%d panoramas of %s in %.1f s: %s, %d threads" % (n, args.workload, dt, what, threads)}

    in_bytes, out_numel, out_pitch = w.in_bytes, int(w.out.numel()), int(w.out.stride(1))
    algo_bytes = w.algo_bytes
    w.free()

    # ---- the other BASELINE configurations ----------------------------------------------
    extra = {}
    if not args.no_extra:
        for name in ("cfg2_6x1080p", "cfg3_8x2160p"):
            if name != args.workload:
                extra[name] = extra_resident(name, device, rank, ctx, world, peak)
        extra["cfg5_sequence"] = extra_sequence(device, rank, world, ctx, args.sequence_frames, args.chunk)
        extra["cfg2_feather_blend"] = extra_blend(device, rank, world, ctx, peak, chunk=args.chunk)
        if rank == 0:
            extra["cfg4_recalibration"] = extra_recalibration(device)
            extra["recorded_capture"] = extra_recorded(device)
            extra["single_call"] = extra_single_call(device)
        barrier()

    ctx.close()
    if rank != 0:
        return
    line = {
        "metric": "panoramas_per_sec", "value": pps, "unit": "panoramas/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic", "output_mp_per_s": pps * out_w * out_h / 1e6,
        "config": {"workload": args.workload, "cameras": n_cams, "frame_hw": [H, W],
                   "panorama_wh": [out_w, out_h], "panoramas_per_launch": batch, "launches_per_step": lps,
                   "panoramas_per_step_per_gpu": batch * lps,
                   "sharding": "frame range per rank, no collective (gloo carries the barrier and two scalars)",
                   "l2": "inputs per launch %.0f MB + outputs %.0f MB per GPU, larger than the 126 MB L2"
                         % (in_bytes / 1e6, out_numel / 1e6),
                   "panorama_pitch_bytes": out_pitch, "kernel_variant": variant, "feather_log2": args.feather,
                   "tiled_ctas_per_sm": ctas, "tiled_work_table": stats},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": recorded_traffic(args.workload, batch),
                     "traffic_source": "ncu dram__bytes_read+write per launch, profiles/r2_dram_traffic.json",
                     "algorithmic_bytes_per_launch": algo_bytes * batch,
                     "launches_per_step": launches // max(args.steps, 1),
                     "peak_source": peak_src,
                     "algorithmic_bytes_per_panorama": algo_bytes,
                     "launch_ms": launch_ms * kernels_per_launch_call, "panoramas_per_launch": batch},
        "cpu_baseline": cpu,
        "e2e": {"value": e2e_pps, "unit": "panoramas/s", "h2d_bytes_per_step": h2d_b * e2e_batch,
                "d2h_bytes_per_step": d2h_b * e2e_batch, "steps": e2e_steps,
                "ms_per_step": e2e_ms / e2e_steps,
                "api": "sequence.SequencePipeline.run(ring=True) (pinned host in/out, %d frame-sets per chunk)" % args.chunk,
                "numa_bound": bool(numa_bound),
                "host_ceiling_gbs": {"h2d": up_gbs, "d2h": dn_gbs,
                                     "how": "all %d ranks at once, plain pinned 256 MB cudaMemcpyAsync both ways" % world},
                "host_ceiling_panoramas_per_s": ceiling_pps, "frac_of_host_ceiling": e2e_pps / ceiling_pps},
        "gpu_launches": launches,
        "clocks": clocks,
        "parity": parity,
        "extra": extra,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="frame-sets per launch per GPU (0 = workload default)")
    ap.add_argument("--launches-per-step", type=int, default=LAUNCHES_PER_STEP)
    ap.add_argument("--whole-frames", action="store_true",
                    help="e2e path uploads whole camera frames instead of the windows the panorama can see")
    ap.add_argument("--chunk", type=int, default=16, help="frame-sets per pipeline chunk of the e2e path")
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU baseline work")
    ap.add_argument("--pitch-align", type=int, default=128, help="row pitch alignment of the device-resident panoramas")
    ap.add_argument("--feather", type=int, default=0, help="feather blend over 2**n pixels (0 = reference overwrite)")
    ap.add_argument("--sequence-frames", type=int, default=10000, help="frames of the config-5 sequence (extra record)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="kernel experiments: skip the end-to-end leg and the extras")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra records (configs 2-5)")
    ap.add_argument("--ref-panos-per-step", type=int, default=4)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a seeded sample of the last timed step's panoramas to DIR/*.npy (rank 0)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
