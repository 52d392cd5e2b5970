"""Recorded-sequence driver: frame-range sharding across GPUs and the pipelined
host -> device -> kernel -> host path.

Every panorama depends only on its own N frames and the fixed calibration
(``Stitcher.stitch`` keeps no state between calls, reference
StitcherClass.py:114-136), so a sequence shards by contiguous frame range with
no data-path collective: each process (one per GPU) composites its range and
only its own output goes back to the host (SURVEY.md section 8 row e).
"""
import torch

from . import _cabi


def shard_range(n_frames, world_size, rank):
    """Contiguous frame range ``[lo, hi)`` of ``rank``: sizes differ by at most
    one, earlier ranks take the remainder, ranges tile ``[0, n_frames)``."""
    if world_size < 1 or not (0 <= rank < world_size):
        raise ValueError("bad rank %d / world size %d" % (rank, world_size))
    base, rem = divmod(int(n_frames), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def ring_chunks(lo, hi, ring, chunk, ramp=False):
    """How frames ``[lo, hi)`` of a sequence held in a ring of ``ring`` host slots (frame ``f`` in slot
    ``f % ring``) are cut into pipeline chunks: ``(slot, n)`` pairs of at most ``chunk`` consecutive
    slots that never wrap around the end of the ring.

    ``ramp=True``: the chunks grow 1, 2, 4, ... up to ``chunk`` at the start and halve towards the end.
    Nothing overlaps the upload of the first chunk or the download of the last one, so with full-size
    chunks a run of ``F`` frames pays about ``2 * chunk / F`` of its transfer time for filling and
    draining the pipeline (13 % for 240 frame-sets in chunks of 16); ramped, about ``2 / F``."""
    out = []
    f = int(lo)
    cap = 1 if ramp else int(chunk)
    while f < hi:
        r0 = f % ring
        n = min(int(chunk), cap, hi - f, ring - r0)
        if ramp:
            n = min(n, max(1, (hi - f + 1) // 2))
            cap = min(int(chunk), cap * 2)
        out.append((r0, n))
        f += n
    return out


def pinned_like(shape, dtype=torch.uint8):
    return torch.empty(shape, dtype=dtype, pin_memory=True)


class SequencePipeline(object):
    """Composite a host-resident sequence chunk by chunk with copies and
    kernels overlapped on three streams (H2D, compute, D2H) and ``depth``
    device-side slots.

    ``run(host_frames, host_out)``: ``host_frames[label]`` is a pinned uint8
    tensor ``[F, H, W, C]``, ``host_out`` a pinned ``[F, H_out, W_out, C]``.
    """

    def __init__(self, stitcher, img_shapes, device, chunk=16, depth=3, windows=True):
        self.stitcher = stitcher
        self.device = torch.device(device)
        self.labels = list(stitcher.img_labels)
        self.plan = stitcher.plan(img_shapes, self.device)
        if self.plan is None:
            raise ValueError("stitcher is not calibrated")
        self.chunk = int(chunk)
        self.depth = int(depth)
        with torch.cuda.device(self.device):
            self.s_in = torch.cuda.Stream()
            self.s_k = torch.cuda.Stream()
            self.s_out = torch.cuda.Stream()
            self.slots = []
            for _ in range(self.depth):
                src = [torch.empty((self.chunk,) + tuple(s), dtype=torch.uint8, device=self.device)
                       for s in img_shapes]
                dst = self.plan.new_output(self.chunk)
                self.slots.append(dict(src=src, dst=dst, ev_in=torch.cuda.Event(), ev_k=torch.cuda.Event(),
                                       ev_out=torch.cuda.Event(), used=False))

        # Host -> device: only the part of every camera that can reach the panorama
        # (CompiledPlan.upload_bands: per band of source rows the column range the kernel reads).
        # What is hidden under the pasted inner canvas is never read and stays whatever the device
        # buffer held.  ``windows=False`` uploads whole frames.
        bands = self.plan.upload_bands(whole=not windows)
        self.windows = []     # per camera: list of copies {b0, nbytes, y0, rows}
        self.geometry = []    # per camera: (row bytes, rows)
        for c, shape in enumerate(img_shapes):
            h, w = int(shape[0]), int(shape[1])
            row = w * (int(shape[2]) if len(shape) == 3 else 1)
            self.geometry.append((row, h))
            self.windows.append(bands[c][2] if c in bands else [])

    def bytes_per_frame(self):
        h2d = sum(w["nbytes"] * w["rows"] for copies in self.windows for w in copies)
        d2h = int(self.slots[0]["dst"][0].numel())
        return h2d, d2h

    def run(self, host_frames, host_out, lo=0, hi=None, ring=False, sync=True):
        """Composite frames ``[lo, hi)`` of the host sequence into
        ``host_out[lo:hi]``; returns the number of panoramas produced.  The
        call returns after the last device->host copy has completed: the host
        blocks on the download stream, so ``host_out`` may be read right away.
        ``sync=False`` only orders the caller's current stream behind the
        pipeline (a device-side dependency, the host does not wait): the caller
        must synchronise that stream before it touches ``host_out``.

        ``ring=True``: the host tensors are rings of ``R`` frame-sets / panoramas and frame ``f``
        of the sequence lives in slot ``f % R`` (a long synthetic sequence cycled through a few
        resident frame-sets, or a capture decoded just ahead of the pipeline); ``[lo, hi)`` may
        then be any range."""
        F = int(host_out.shape[0])
        hi = F if hi is None else hi
        if ring:
            return self._run_ring(host_frames, host_out, int(lo), int(hi), F, sync)
        with torch.cuda.device(self.device):
            start = torch.cuda.current_stream()
            for s in (self.s_in, self.s_k, self.s_out):
                s.wait_stream(start)
            # one "ring" as long as the sequence: the same ramped schedule, no wrap-around
            for i, (f0, n) in enumerate(ring_chunks(lo, hi, max(F, hi), self.chunk, ramp=True)):
                self._chunk(i, host_frames, host_out, f0, n)
            self._finish(start, sync)
        return hi - lo

    def _finish(self, start, sync):
        start.wait_stream(self.s_out)
        start.wait_stream(self.s_k)
        start.wait_stream(self.s_in)
        if sync:
            # the last chunk's download is the last operation of s_out, and every kernel and upload precedes one
            self.s_out.synchronize()

    def _chunk(self, i, host_frames, host_out, f0, n):
        """Enqueue chunk ``i``: host frames ``[f0, f0 + n)`` -> slot -> kernel -> ``host_out[f0:f0 + n]``."""
        slot = self.slots[i % self.depth]
        with torch.cuda.stream(self.s_in):
            if slot["used"]:
                self.s_in.wait_event(slot["ev_k"])      # previous kernel done reading the slot
            for c, label in enumerate(self.labels):
                host = host_frames[label]
                row, h = self.geometry[c]
                copies = self.windows[c]
                if len(copies) == 1 and copies[0]["nbytes"] == row and copies[0]["rows"] == h:
                    slot["src"][c][:n].copy_(host[f0:f0 + n], non_blocking=True)
                    continue
                if copies and not host.is_contiguous():
                    raise ValueError("host frames of %r must be contiguous" % (label,))
                fs = row * h
                for w in copies:
                    _cabi.copy_window_u8(slot["src"][c].data_ptr(), row, fs, host.data_ptr() + f0 * fs, row, fs,
                                         w["b0"], w["nbytes"], w["y0"], w["rows"], n, self.s_in.cuda_stream)
            slot["ev_in"].record(self.s_in)
        with torch.cuda.stream(self.s_k):
            self.s_k.wait_event(slot["ev_in"])
            if slot["used"]:
                self.s_k.wait_event(slot["ev_out"])     # previous D2H done reading dst
            self.plan.run([t[:n] for t in slot["src"]], out=slot["dst"][:n], n_frames=n,
                          stream=self.s_k)
            slot["ev_k"].record(self.s_k)
        with torch.cuda.stream(self.s_out):
            self.s_out.wait_event(slot["ev_k"])
            host_out[f0:f0 + n].copy_(slot["dst"][:n], non_blocking=True)
            slot["ev_out"].record(self.s_out)
        slot["used"] = True

    def _run_ring(self, host_frames, host_out, lo, hi, R, sync=True):
        with torch.cuda.device(self.device):
            start = torch.cuda.current_stream()
            for s in (self.s_in, self.s_k, self.s_out):
                s.wait_stream(start)
            for i, (r0, n) in enumerate(ring_chunks(lo, hi, R, self.chunk, ramp=True)):
                self._chunk(i, host_frames, host_out, r0, n)
            self._finish(start, sync)
        return hi - lo
