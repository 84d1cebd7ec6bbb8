"""Host logic of the CuMemAllocator mirror on CPU, with a recording engine injected: argument normalisation is the
reference's (cumem.py:186-194), tiers/knobs come from the environment, and the INFO line the reference's benchmark
tooling parses (cumem.py:215-222; inference_server/benchmark/benchmark.md:157) keeps its wording."""
import logging
import os
import re

import pytest

import fma_b200  # noqa: F401
from fma_b200 import _lib as L
from fma_b200 import cumem
from fma_b200.engine import SegmentInfo

GiB = 1 << 30


class FakeEngine:
    def __init__(self):
        self.calls = []
        self.segs = [SegmentInfo(0, 0x7000000000, 15 * GiB, 15 * GiB, None, 0, "weights", True, False, 0),
                     SegmentInfo(1, 0x9000000000, 32 * GiB, 32 * GiB, None, 1, "kv_cache", True, False, 0)]

    def make_current(self): self.calls.append(("make_current",))
    def segments(self): return self.segs
    def current_usage(self): return sum(s.bytes for s in self.segs)
    def sleep(self, offload, tier=0, flags=0): self.calls.append(("sleep", tuple(offload), tier))
    def wake(self, tags, flags=0): self.calls.append(("wake", tags))
    def peer_reserve(self, dev, n): self.calls.append(("peer_reserve", dev, n))
    def host_reserve(self, n): self.calls.append(("host_reserve", n))

    def stats(self):
        return {"sleep_bytes_offloaded": 15 * GiB, "sleep_bytes_discarded": 32 * GiB, "sleep_copy_seconds": 0.28, "sleep_seconds": 0.29,
                "wake_bytes_restored": 15 * GiB, "wake_copy_seconds": 0.29, "wake_seconds": 0.2925}


@pytest.fixture()
def alloc(monkeypatch):
    for k in ("FMA_TIER", "FMA_PEER_DEVICE"):
        monkeypatch.delenv(k, raising=False)
    return cumem.CuMemAllocator(engine=FakeEngine())


def test_offload_tag_normalisation_matches_the_reference(alloc):
    alloc.sleep()                                   # None -> (default_tag,)
    alloc.sleep("weights")                          # str -> 1-tuple
    alloc.sleep(offload_tags=("weights",))          # what Worker.sleep(level=1) passes
    alloc.sleep(offload_tags=tuple())               # level 2
    got = [c for c in alloc.engine.calls if c[0] == "sleep"]
    assert got == [("sleep", ("default",), L.FMA_TIER_HOST), ("sleep", ("weights",), L.FMA_TIER_HOST),
                   ("sleep", ("weights",), L.FMA_TIER_HOST), ("sleep", (), L.FMA_TIER_HOST)]
    with pytest.raises(AssertionError):
        alloc.sleep(offload_tags=["weights"])       # the reference asserts a tuple too (cumem.py:196)
    alloc.wake_up(); alloc.wake_up(tags=["weights"])
    assert [c for c in alloc.engine.calls if c[0] == "wake"] == [("wake", None), ("wake", ["weights"])]


def test_reference_log_line_wording(alloc, caplog):
    with caplog.at_level(logging.INFO, logger="vllm.fma_b200.cumem"):
        alloc.sleep(offload_tags=("weights",))
    msg = "\n".join(r.getMessage() for r in caplog.records)
    m = re.search(r"CuMemAllocator: sleep freed ([\d.]+) GiB memory in total, of which ([\d.]+) GiB is backed up in CPU and the "
                  r"rest ([\d.]+) GiB is discarded directly\.", msg)
    assert m and [float(x) for x in m.groups()] == [47.0, 15.0, 32.0]
    assert "D2H" in msg


def test_registry_view_and_usage(alloc):
    ptd = alloc.pointer_to_data
    assert set(ptd) == {0x7000000000, 0x9000000000}
    d = ptd[0x7000000000]
    assert d.handle[:3] == (0, 15 * GiB, 0x7000000000) and d.tag == "weights" and d.cpu_backup_tensor is None
    assert alloc.get_current_usage() == 47 * GiB


def test_peer_tier_comes_from_the_environment(alloc, monkeypatch):
    monkeypatch.setenv("FMA_TIER", "peer")
    with pytest.raises(L.FmaError):
        alloc.sleep(offload_tags=("weights",))      # no parking device named
    monkeypatch.setenv("FMA_PEER_DEVICE", "5")
    alloc.sleep(offload_tags=("weights",))
    assert ("peer_reserve", 5, 15 * GiB) in alloc.engine.calls
    assert alloc.engine.calls[-1] == ("sleep", ("weights",), L.FMA_TIER_PEER)

    def no_room(dev, n):
        raise L.FmaError(L.FMA_ENOMEM, "cuMemCreate(peer store) failed: out of memory")
    monkeypatch.setattr(alloc.engine, "peer_reserve", no_room)          # the parking GPU is full right now: the sleep goes to the host tier
    alloc.sleep(offload_tags=("weights",))
    assert alloc.engine.calls[-1] == ("sleep", ("weights",), L.FMA_TIER_HOST)

    def broken(dev, n):
        raise L.FmaError(L.FMA_ECUDA, "no NVLink path")
    monkeypatch.setattr(alloc.engine, "peer_reserve", broken)           # anything else stays loud
    with pytest.raises(L.FmaError):
        alloc.sleep(offload_tags=("weights",))


def test_peer_tier_falls_back_to_the_host_tier_when_no_gpu_can_take_the_image(alloc, monkeypatch, sock_dir, caplog):
    """Under the node agent the parking buffer is the agent's (parking.py).  If every candidate GPU is full — or the agent is gone —
    the sleep still has to succeed: it goes to the host tier, as the reference's always does (cumem.py:237-249), and says so."""
    from fma_b200.parking import ParkingService

    def full(device, nbytes):
        raise MemoryError(f"cuMemCreate on device {device}: out of memory")

    sock = os.path.join(sock_dir, "agent.sock")
    svc = ParkingService(sock, n_devices=4, make_buffer=full)
    svc.start()
    monkeypatch.setenv("FMA_TIER", "peer")
    monkeypatch.setenv("FMA_NODE_AGENT_SOCK", sock)
    monkeypatch.setenv("FMA_NODE_GPU_INDICES", "0")
    try:
        with caplog.at_level(logging.WARNING, logger="vllm.fma_b200.cumem"):
            alloc.sleep(offload_tags=("weights",))
        assert alloc.engine.calls[-1] == ("sleep", ("weights",), L.FMA_TIER_HOST)
        assert any("sleeping to the host tier instead" in r.getMessage() and "no GPU can take 15360 MiB" in r.getMessage() for r in caplog.records)
        assert svc.stats()["images"] == []
    finally:
        svc.close()
    alloc.engine.calls.clear()
    alloc.sleep(offload_tags=("weights",))          # the agent's socket is gone altogether
    assert alloc.engine.calls[-1] == ("sleep", ("weights",), L.FMA_TIER_HOST)
