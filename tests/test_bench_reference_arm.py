"""The reference arm of ``bench.py`` (``--impl reference``) runs on host cores only, so it is checked here: one
JSON line with the contract's keys, the reference's own ``Stitcher`` class behind it where the build output
``oracle/_ref`` can be made or found, and a silent exit 0 for the ranks other than 0."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None, args=()):
    env = dict(os.environ)
    env.update(extra_env or {})
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg1_3x720p",
                        "--steps", "2", "--warmup", "1", "--ref-panos-per-step", "1"] + list(args),
                       cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert r.returncode == 0, r.stderr.decode(errors="replace")[-2000:]
    return r.stdout.decode().strip().splitlines()


@pytest.mark.parametrize("port", [False, True])
def test_reference_arm_line(port):
    from oracle import build_ref
    lines = _run({"MCS_BENCH_REFERENCE_PORT": "1"} if port else None)
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "panoramas_per_sec" and d["unit"] == "panoramas/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1
    assert d["value"] > 0 and d["gpu_launches"] == 0 and d["vs_baseline"] is None and d["dtype"] == "u8"
    assert d["config"]["workload"] == "cfg1_3x720p" and d["config"]["panoramas_per_step"] == 1
    assert d["e2e"] == {"value": d["value"], "unit": "panoramas/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["value"] == d["value"] and cb["cores"] >= 1 and cb["sample"]
    have_ref = build_ref.available() or build_ref.prebuilt() is not None
    assert cb["kind"] == ("reference" if have_ref and not port else "port")


def _chain_panoramas(frame_indices):
    """The cv2 chain's panoramas of the cfg1_3x720p workload for the given synthetic frame indices."""
    import numpy as np
    from multicamera_stitching_b200 import synthetic
    from oracle import stitcher_ref
    st, homographies, labels, images = synthetic.synthetic_stitcher(3, 720, 1280, 3, kind="smooth")
    states = stitcher_ref.calibrate_chain_from_homographies([images[l].shape for l in labels], homographies)
    return np.stack([stitcher_ref.stitch_chain(states, labels, synthetic.make_frames(3, 720, 1280, 3, frame_index=f,
                                                                                     kind="smooth"))
                     for f in frame_indices])


def _load_dump(d, name):
    import numpy as np
    vals, pix = np.load(os.path.join(str(d), name + ".npy")), np.load(os.path.join(str(d), name + "_pixels.npy"))
    assert vals.dtype == pix.dtype == np.float32 and pix.shape == (len(vals), 3) and len(vals) > 0
    return vals, pix.astype(np.int64)


def test_reference_arm_dumps_its_last_step(tmp_path):
    """``--dump-outputs`` plumbing of the CPU arm: float32 files within 64 MB, the same on every run with the same
    arguments, holding the last step's panorama at the sampled pixels.  The expected panorama comes from the cv2
    chain, which is also what this arm runs where ``oracle/_ref`` is absent, so this checks the dump, not the chain."""
    import numpy as np
    dumps = []
    for k in range(2):
        _run(args=["--dump-outputs", str(tmp_path / str(k))])
        dumps.append(_load_dump(tmp_path / str(k), "panoramas"))
        total = sum(os.path.getsize(os.path.join(str(tmp_path / str(k)), n)) for n in os.listdir(str(tmp_path / str(k))))
        assert total <= 64 << 20
    (vals, pix), (vals2, pix2) = dumps
    assert np.array_equal(vals, vals2) and np.array_equal(pix, pix2)
    want = _chain_panoramas([0])      # one panorama per step: frame-set 0
    assert np.array_equal(vals, want[pix[:, 0], pix[:, 1], pix[:, 2]].astype(np.float32))


@pytest.mark.gpu
def test_gpu_arm_dumps_its_last_step(cuda_device, tmp_path):
    """``--dump-outputs`` of the GPU arm: the timed launches' and the end-to-end leg's panoramas at the sampled pixels
    equal the cv2 chain's within the bench's own parity bound, and ``--steps`` sets the steps of both legs.  The bench
    zeroes both outputs after their warm-up, so the values checked here were written by the timed steps."""
    import numpy as np
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg1_3x720p", "--batch", "2",
                        "--steps", "2", "--warmup", "1", "--launches-per-step", "1", "--no-cpu", "--no-extra",
                        "--dump-outputs", str(tmp_path)],
                       cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert r.returncode == 0, r.stderr.decode(errors="replace")[-2000:]
    d = json.loads(r.stdout.decode().strip().splitlines()[-1])
    assert d["steps"] == 2 and d["e2e"]["steps"] == 2
    want = _chain_panoramas([0, 1])   # batch of 2: frame-set f is synthetic frame index f
    for name in ("panoramas", "e2e_panoramas"):
        vals, pix = _load_dump(tmp_path, name)
        diff = np.abs(vals - want[pix[:, 0], pix[:, 1], pix[:, 2]])
        assert diff.max() <= 1 and (diff == 0).mean() >= 0.999, name


def test_other_ranks_print_nothing():
    assert _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}, ["--gpus", "2"]) == []


def test_gpu_arm_refuses_to_run_without_a_device():
    """No CPU fallback: without a CUDA device the GPU arm ends with an error instead of a number."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], cwd=ROOT,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert r.returncode != 0 and r.stdout.decode().strip() == ""
    assert "no CUDA device" in r.stderr.decode(errors="replace")
