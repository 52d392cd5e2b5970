"""Host model of the tiled kernel's producer protocol (csrc/mcs_stitch_tiled.cu: ``produce`` and the consumer loop
of ``mcs_stitch_tiled_kernel``), run over random chunk sequences and random interleavings.

One producer thread claims chunks, publishes their ids into a ring of TILED_QD entries, copies each chunk's record
into one of two buffers and issues every staged box into a ring of `stages` slots.  Eight resampling warps read the
ids, wait for the records and boxes, and release both.  Every handshake is an mbarrier wait on a phase parity, so
a slot or buffer that is refilled early, or a wait that is never satisfied, does not fault: it hangs the CTA or
resamples the wrong box.  The model keeps the kernel's barriers (phase counts, parity waits, arrival counts,
transfers that land at a random later time) and its order of operations, lets the actors run in a random order,
and checks that no run deadlocks, that no slot, record buffer or id entry is overwritten before every warp is done
with it, and that every warp reads the box, record and id it expects.  It is a model of the protocol, not of the
arithmetic; the GPU tests hold the kernel itself."""
import random

import pytest

ZERO, COPY, WARP, BAND = 0, 1, 2, 4
QD = 32            # TILED_QD
WARPS = 8          # TILED_WARPS


class Deadlock(Exception):
    pass


class Barrier(object):
    """An mbarrier: a phase completes when `count` arrivals and the expected transfers are in."""

    def __init__(self, count):
        self.count = count
        self.arrived = 0
        self.phase = 0             # completed phases

    def arrive(self):
        self.arrived += 1
        assert self.arrived <= self.count, "more arrivals than the barrier counts"
        if self.arrived == self.count:
            self.arrived = 0
            self.phase += 1

    def passed(self, parity):      # mbarrier.try_wait.parity / test_wait.parity
        return (self.phase & 1) != parity


class Cta(object):
    def __init__(self, chunks, stages, claim, rng, producer=None):
        self.chunks = chunks                       # this CTA's chunks in claim order; the end marker follows
        self.stages = stages
        self.claim = claim
        self.rng = rng
        self.full = [Barrier(1) for _ in range(stages)]
        self.empty = [Barrier(WARPS) for _ in range(stages)]
        self.slot_box = [None] * stages            # what the TMA wrote into each slot
        self.slot_readers = [set() for _ in range(stages)]
        self.rec_full = [Barrier(1) for _ in range(2)]
        self.rec_empty = [Barrier(WARPS) for _ in range(2)]
        self.rec_buf = [None, None]
        self.rec_readers = [set(), set()]
        self.ov_full, self.ov_empty = Barrier(1), Barrier(WARPS)
        self.ids = [None] * QD
        self.published = 0
        self.next_id = [0] * WARPS                 # sequence number each warp reads next
        self.landing = []                          # transfers in flight: (barrier, action)
        self.producer = producer or produce

    # -- what the chunk sequence says --------------------------------------------------------------
    def boxes(self, k):
        """The boxes of chunk k in issue (= consumption) order: (chunk, frame, box index)."""
        ch = self.chunks[k]
        if ch["cls"] == ZERO:
            return []
        first = 1 if ch.get("zero_base") else 0
        per_frame = range(first, 1 + ch.get("n_ov", 0)) if ch["cls"] == BAND else [0]
        return [(k, f, li) for f in range(ch["frames"]) for li in per_frame]

    # -- transfers (TMA box, bulk copy of a record, overlay descriptors) -----------------------------
    def start_transfer(self, bar, action):
        assert all(b is not bar for b, _ in self.landing), "a second transfer on a barrier whose phase has not completed"
        self.landing.append((bar, action))

    def land_one(self):
        bar, action = self.landing.pop(self.rng.randrange(len(self.landing)))
        action()
        bar.arrive()

    # -- the producer's pieces -------------------------------------------------------------------------
    def publish(self, j):
        """sched_ensure writing sequence number j into the id ring."""
        assert all(n > j - QD for n in self.next_id), "id entry %d overwritten before every warp read it" % (j - QD)
        self.ids[j % QD] = j if j < len(self.chunks) else -1
        self.published = j + 1

    def prefetch(self, b, k):
        assert self.rec_buf[b] is None or len(self.rec_readers[b]) == WARPS, \
            "record buffer %d refilled while a warp still reads it" % b
        def land():
            self.rec_buf[b] = k
            self.rec_readers[b] = set()
        self.start_transfer(self.rec_full[b], land)

    def issue(self, slot, box):
        assert self.slot_box[slot] is None or len(self.slot_readers[slot]) == WARPS, \
            "slot %d overwritten before every warp released box %r" % (slot, self.slot_box[slot])
        def land():
            self.slot_box[slot] = box
            self.slot_readers[slot] = set()
        self.start_transfer(self.full[slot], land)

    def run(self, max_steps=10 ** 6):
        actors = [self.producer(self)] + [consume(self, w) for w in range(WARPS)]
        waits = [None] * len(actors)                       # condition each actor blocks on
        live = list(range(len(actors)))
        for _ in range(max_steps):
            ready = [i for i in live if waits[i] is None or waits[i]()]
            choices = len(ready) + (1 if self.landing else 0)
            if choices == 0:
                if not live:
                    assert not self.landing
                    return
                raise Deadlock("no actor can move: producer %s, warps at chunks %r"
                               % ("done" if 0 not in live else "blocked", self.next_id))
            pick = self.rng.randrange(choices)
            if pick == len(ready):
                self.land_one()
                continue
            i = ready[pick]
            try:
                waits[i] = next(actors[i])
            except StopIteration:
                live.remove(i)
        raise AssertionError("the model did not finish")


def produce(cta):
    """``produce<BANDS>``: yields the condition it waits on."""
    st = dict(claimed=0)

    def sched_ensure(upto):
        while st["claimed"] < upto and st["claimed"] <= len(cta.chunks):
            for _ in range(cta.claim):
                if st["claimed"] > len(cta.chunks):
                    break
                cta.publish(st["claimed"])
                st["claimed"] += 1

    sched_ensure(1)
    if cta.ids[0] >= 0:
        cta.prefetch(0, 0)
    slot, phase = 0, 0
    k = 0
    while True:
        sched_ensure(k + 2)
        if cta.ids[k % QD] < 0:
            break
        assert cta.ids[k % QD] == k
        rec_todo = cta.ids[(k + 1) % QD] >= 0
        b, rel_par = (k + 1) & 1, ((k - 1) >> 1) & 1
        for box in cta.boxes(k):
            if rec_todo and (k == 0 or cta.rec_empty[b].passed(rel_par)):
                cta.prefetch(b, k + 1)
                rec_todo = False
            yield (lambda s=slot, p=phase: cta.empty[s].passed(p ^ 1))
            cta.issue(slot, box)
            slot += 1
            if slot == cta.stages:
                slot, phase = 0, phase ^ 1
        if rec_todo:
            if k >= 1:
                yield (lambda: cta.rec_empty[b].passed(rel_par))
            cta.prefetch(b, k + 1)
        k += 1


def consume(cta, w):
    """One resampling warp of ``mcs_stitch_tiled_kernel``."""
    slot, phase = 0, 0
    band_seq = 0
    k = 0
    while True:
        yield (lambda: cta.published > k)
        j = cta.ids[k % QD]
        cta.next_id[w] = k + 1
        if j < 0:
            return
        assert j == k, "warp %d read id %r for chunk %d" % (w, j, k)
        cb = k & 1
        yield (lambda: cta.rec_full[cb].passed((k >> 1) & 1))
        assert cta.rec_buf[cb] == k, "warp %d found the record of chunk %r for chunk %d" % (w, cta.rec_buf[cb], k)
        ch = cta.chunks[k]
        if ch["cls"] == BAND:
            if w == 0:
                if band_seq > 0:
                    yield (lambda s=band_seq: cta.ov_empty.passed((s - 1) & 1))
                cta.start_transfer(cta.ov_full, lambda: None)
            yield (lambda s=band_seq: cta.ov_full.passed(s & 1))
        cta.rec_readers[cb].add(w)
        cta.rec_empty[cb].arrive()
        for box in cta.boxes(k):
            yield (lambda s=slot, p=phase: cta.full[s].passed(p))
            assert cta.slot_box[slot] == box, "warp %d expected box %r, slot %d holds %r" % (w, box, slot, cta.slot_box[slot])
            cta.slot_readers[slot].add(w)
            cta.empty[slot].arrive()
            slot += 1
            if slot == cta.stages:
                slot, phase = 0, phase ^ 1
        if ch["cls"] == BAND:
            band_seq += 1
            cta.ov_empty.arrive()
        k += 1


def random_sweep(rng, with_bands, split, last_frames):
    """One CTA's chunks: runs of ZERO chunks, BAND chunks (zero-base ones too), split chunks of a few frames, a last
    frame block of `last_frames` frames."""
    n = rng.randint(0, 40)
    block = rng.choice([4, 8, 16, 64])
    chunks = []
    for blk, nf in ((0, block), (1, last_frames)):
        for i in range(n):
            r = rng.random()
            parts = split if r < 0.3 else 1
            cls = BAND if with_bands and r < 0.2 else WARP if r < 0.45 else COPY if r < 0.6 else ZERO
            for p in range(parts):
                frames = nf * (p + 1) // parts - nf * p // parts
                ch = dict(cls=cls, frames=frames)
                if cls == BAND:
                    ch.update(n_ov=rng.choice([1, 2]), zero_base=rng.random() < 0.3)
                chunks.append(ch)
            if cls == ZERO and rng.random() < 0.3:     # a run of ZERO chunks
                chunks.extend(dict(cls=ZERO, frames=nf) for _ in range(rng.randint(1, 12)))
    # this CTA's share: a random subsequence, as the claims of the other CTAs leave it
    return [c for c in chunks if rng.random() < 0.7]


@pytest.mark.parametrize("with_bands", [False, True])
@pytest.mark.parametrize("split", [1, 4])
@pytest.mark.parametrize("last_frames", [1, 2, 3, 64])
def test_no_deadlock_and_no_early_overwrite(with_bands, split, last_frames):
    rng = random.Random(7 + 100 * with_bands + 10 * split + last_frames)
    for _ in range(60):
        chunks = random_sweep(rng, with_bands, split, last_frames)
        Cta(chunks, rng.choice([3, 4, 6, 7, 8]), rng.randint(1, 8), rng).run()


def test_end_marker_alone_and_right_after_one_chunk():
    rng = random.Random(5)
    Cta([], 4, 1, rng).run()
    for cls in (ZERO, COPY, WARP, BAND):
        Cta([dict(cls=cls, frames=3, n_ov=2)], 3, rng.randint(1, 8), rng).run()


def test_chunks_without_frames_do_not_hang():
    """A split tile cut into more parts than a short block has frames gives chunks with no frames; the producer
    steps over them like ZERO chunks."""
    rng = random.Random(11)
    chunks = [dict(cls=WARP, frames=2)] + [dict(cls=WARP, frames=0)] * 5 + [dict(cls=COPY, frames=1)]
    for _ in range(50):
        Cta(chunks, 3, rng.randint(1, 8), rng).run()


def test_the_model_catches_a_record_copied_before_its_buffer_is_released():
    def eager(cta):
        # what the release wait prevents: the next record goes into its buffer at once
        slot, phase, k = 0, 0, 0
        for j in range(len(cta.chunks) + 1):
            cta.publish(j)
        if cta.chunks:
            cta.prefetch(0, 0)
        for k in range(len(cta.chunks)):
            if k + 1 < len(cta.chunks):
                cta.prefetch((k + 1) & 1, k + 1)
            for box in cta.boxes(k):
                yield (lambda s=slot, p=phase: cta.empty[s].passed(p ^ 1))
                cta.issue(slot, box)
                slot += 1
                if slot == cta.stages:
                    slot, phase = 0, phase ^ 1
    chunks = [dict(cls=WARP, frames=2) for _ in range(6)]
    with pytest.raises(AssertionError):
        for seed in range(20):
            Cta(chunks, 4, 1, random.Random(seed), producer=eager).run()


def test_the_model_catches_a_box_issued_without_its_slot_wait():
    def hasty(cta):
        for j in range(len(cta.chunks) + 1):
            cta.publish(j)
        if cta.chunks:
            cta.prefetch(0, 0)
        slot = 0
        for k in range(len(cta.chunks)):
            for box in cta.boxes(k):
                yield None
                cta.issue(slot, box)
                slot = (slot + 1) % cta.stages
            if k + 1 < len(cta.chunks):
                b = (k + 1) & 1
                if k >= 1:
                    yield (lambda: cta.rec_empty[b].passed(((k - 1) >> 1) & 1))
                cta.prefetch(b, k + 1)
    chunks = [dict(cls=WARP, frames=8)]
    with pytest.raises(AssertionError):
        for seed in range(20):
            Cta(chunks, 3, 1, random.Random(seed), producer=hasty).run()
