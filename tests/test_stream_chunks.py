"""CPU tests of `distributed.stream_chunks` with fake jobs: the ring of result buffers (one per job in flight) and the draining of
jobs still in flight when a submit, a wait or `on_done` raises."""
import numpy as np
import pytest

from metagenomic_deepfri_b200 import distributed

C = 3


class FakeJob:
    """Writes chunk k's scores at wait(); `log` records submits and waits in order."""

    def __init__(self, k, rows, log, fail=False):
        self.k, self.rows, self.log, self.fail, self.done = k, rows, log, fail, False
        log.append(("submit", k))

    def wait(self):
        assert not self.done
        self.done = True
        self.log.append(("wait", self.k))
        if self.fail:
            raise ValueError(f"job {self.k} failed")
        self.rows[...] = self.k * 100 + np.arange(len(self.rows))[:, None] + np.zeros((1, C))


def sizes():
    return [5, 7, 2, 7, 1, 6]


def test_ring_holds_only_the_chunks_in_flight():
    log, jobs, seen = [], [], {}
    ring = [np.full((7, C), -1.0, np.float32) for _ in range(2)]

    def on_done(k, rows):
        assert np.shares_memory(rows, ring[k % 2]) and len(rows) == sizes()[k]
        seen[k] = rows.copy()

    def submit(k, rows):
        # at most one other job is in flight when a chunk is submitted, and the chunk two back has been written out
        assert sum(1 for j in jobs if not j.done) <= 1 and (k < 2 or k - 2 in seen)
        jobs.append(FakeJob(k, rows, log))
        return jobs[-1]
    distributed.stream_chunks(submit, ((k, n) for k, n in enumerate(sizes())), ring, on_done=on_done)
    assert sorted(seen) == list(range(len(sizes())))
    for k, n in enumerate(sizes()):
        assert np.array_equal(seen[k], k * 100 + np.arange(n)[:, None] + np.zeros((1, C)))
    assert all(j.done for j in jobs)


def test_ring_shape_errors():
    with pytest.raises(ValueError, match="exactly depth"):
        distributed.stream_chunks(lambda c, rows: None, [(0, 1)], [np.zeros((4, C), np.float32)] * 3)
    log = []
    with pytest.raises(ValueError, match="chunk 1 has 9 rows"):
        distributed.stream_chunks(lambda k, rows: FakeJob(k, rows, log), [(0, 3), (1, 9)], [np.zeros((4, C), np.float32)] * 2)
    assert ("wait", 0) in log                                   # chunk 0 was in flight: drained


def test_jobs_in_flight_are_drained_when_a_submit_raises():
    log = []

    def submit(k, rows):
        if k == 3:
            raise ValueError("bad chunk 3")
        return FakeJob(k, rows, log, fail=(k == 2))             # chunk 2's own error is dropped while draining
    out = np.zeros((sum(sizes()), C), np.float32)
    with pytest.raises(ValueError, match="bad chunk 3"):
        distributed.stream_chunks(submit, ((k, n) for k, n in enumerate(sizes())), out)
    assert log == [("submit", 0), ("submit", 1), ("wait", 0), ("submit", 2), ("wait", 1), ("wait", 2)]


def test_jobs_in_flight_are_drained_when_on_done_raises():
    log, jobs = [], []

    def on_done(k, rows):
        if k == 1:
            raise RuntimeError("writer failed")

    def submit(k, rows):
        jobs.append(FakeJob(k, rows, log))
        return jobs[-1]
    with pytest.raises(RuntimeError, match="writer failed"):
        distributed.stream_chunks(submit, ((k, n) for k, n in enumerate(sizes())), np.zeros((sum(sizes()), C), np.float32),
                                  on_done=on_done)
    assert all(j.done for j in jobs) and len(jobs) == 3
