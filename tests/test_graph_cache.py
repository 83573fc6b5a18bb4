"""ops.GraphCache, the CUDA-graph policy that FusedTrainer.step and BiGCN's inference share, driven by a fake capture:
enqueue on a batch's first sighting, capture on the second, replay afterwards; captures valid while their pins are
the same objects; FIFO eviction at max_graphs; a bounded first-sighting table that clear() keeps."""
from bigcn_b200.ops import GraphCache


class FakeGraph:
    def __init__(self, log, name):
        self.log, self.name = log, name

    def replay(self):
        self.log.append(("replay", self.name))


class Batch:
    """stands in for a batch object (weakly referenced by the first-sighting table)"""


def make_cache(max_graphs=4, max_seen=64):
    log = []

    def capture(enqueue):
        g = FakeGraph(log, sum(e[0] == "captured" for e in log))
        enqueue()
        return g

    return GraphCache(max_graphs, max_seen, capture=capture), log


def step(cache, log, key, data, pins=()):
    """what the callers do with a batch: replay its capture, else enqueue it on a first sighting, else capture it"""
    if cache.replay(key, pins) is not None:
        return "replay"
    if cache.first_sighting(key, data):
        return "enqueue"
    cache.capture(key, lambda: log.append(("captured", key)), {"key": key}, pins, data)
    return "capture"


def test_first_sighting_enqueues_then_capture_then_replays():
    cache, log = make_cache()
    d = Batch()
    assert [step(cache, log, "k", d) for _ in range(4)] == ["enqueue", "capture", "replay", "replay"]
    assert log == [("captured", "k"), ("replay", 0), ("replay", 0), ("replay", 0)]   # a capture replays once
    assert cache.captures == 1 and cache.replays == 3 and len(cache) == 1
    assert cache.replay("k") == {"key": "k"}                    # the plan of the capture
    other = Batch()
    assert step(cache, log, "k2", other) == "enqueue"
    assert step(cache, log, "k2", d) == "enqueue"      # another object under a key seen once: a first sighting again
    assert step(cache, log, "k2", d) == "capture"


def test_changed_pin_invalidates_the_capture():
    cache, log = make_cache()
    d, ws, ws2, prep = Batch(), object(), object(), object()
    assert [step(cache, log, "k", d, (ws, prep)) for _ in range(3)] == ["enqueue", "capture", "replay"]
    assert cache.replay("k", (ws2, prep)) is None
    assert cache.replay("k", (ws,)) is None
    assert cache.replays == 2
    assert step(cache, log, "k", d, (ws2, prep)) == "capture"    # seen before: captured again at once
    assert cache.replay("k", (ws, prep)) is None and cache.replay("k", (ws2, prep)) is not None
    assert cache.captures == 2 and len(cache) == 1


def test_fifo_eviction_at_max_graphs():
    cache, log = make_cache(max_graphs=2)
    ds = [Batch() for _ in range(3)]
    for i, d in enumerate(ds):
        assert [step(cache, log, i, d) for _ in range(2)] == ["enqueue", "capture"]
    assert len(cache) == 2 and cache.captures == 3
    assert cache.replay(0) is None and cache.replay(1) is not None and cache.replay(2) is not None
    assert step(cache, log, 0, ds[0]) == "capture"               # evicted, still sighted: captured again
    assert cache.replay(1) is None and cache.replay(2) is not None   # the oldest capture went, replays do not refresh


def test_clear_keeps_first_sightings():
    cache, log = make_cache()
    d = Batch()
    assert [step(cache, log, "k", d) for _ in range(2)] == ["enqueue", "capture"]
    cache.clear()
    assert len(cache) == 0 and cache.replay("k") is None
    assert cache.captures == 1 and cache.replays == 1            # the counters count on
    assert step(cache, log, "k", d) == "capture"
    assert cache.captures == 2 and cache.replays == 2


def test_first_sighting_table_is_bounded():
    cache, log = make_cache(max_seen=2)
    ds = [Batch() for _ in range(3)]
    assert [cache.first_sighting(i, d) for i, d in enumerate(ds)] == [True, True, True]   # the third empties the table
    assert cache.first_sighting(2, ds[2]) is False
    assert cache.first_sighting(0, ds[0]) is True
