"""ParkingService bookkeeping without any engine: placement (least-loaded GPU outside `avoid`), re-use of a buffer that is large enough,
accounting in MiB per GPU (what a sleeper budget reads, inference-server.go:1609-1636), lookups before a deposit, release, and the wire
protocol over the unix socket with fds in the ancillary data — a fake buffer factory stands in for fma_b200.ParkingBuffer."""
import os
import tempfile

import fma_b200  # noqa: F401
from fma_b200.parking import MiB, ParkingClient, ParkingService


class FakeBuffer:
    made = []
    full = set()            # GPUs whose HBM an awake instance has filled: creating a buffer there fails

    def __init__(self, device, nbytes):
        if device in FakeBuffer.full:
            raise MemoryError(f"cuMemCreate on device {device}: out of memory")
        self.device, self.nbytes = device, (nbytes + 2 * MiB - 1) // (2 * MiB) * (2 * MiB)
        self._f = tempfile.TemporaryFile()
        self._f.truncate(self.nbytes)
        self.closed = False
        FakeBuffer.made.append(self)

    def export_fd(self):
        return os.dup(self._f.fileno())

    def close(self):
        self.closed = True
        self._f.close()


class FakeEngine:
    def __init__(self):
        self.attached = None

    def peer_attach(self, fd, nbytes):
        assert os.fstat(fd).st_size == nbytes
        self.attached = nbytes

    def image_describe(self, tier):
        return b"DESC" + bytes([tier])

    def image_adopt_parked(self, desc, tags):
        self.adopted = (desc, tuple(tags))


def test_placement_accounting_and_protocol(sock_dir):
    FakeBuffer.made.clear()
    svc = ParkingService(os.path.join(sock_dir, "s.sock"), n_devices=4, make_buffer=FakeBuffer)
    svc.start()
    try:
        cli = ParkingClient(os.path.join(sock_dir, "s.sock"))
        e = FakeEngine()
        r = cli.park(e, "Ia", 0, 100 * MiB, avoid=[0])
        assert r["device"] == 1 and e.attached == 100 * MiB                    # least-loaded GPU outside `avoid`, lowest index first
        assert cli.park(FakeEngine(), "Ib", 0, 50 * MiB, avoid=[0])["device"] == 2    # GPU 1 now carries 100 MiB
        assert cli.park(FakeEngine(), "Ic", 0, 10 * MiB, avoid=[0, 2])["device"] == 3
        assert cli.park(FakeEngine(), "Id", 0, 10 * MiB, device=0)["device"] == 0    # an explicit device wins
        st = cli.stats()
        assert st["parked_mib_per_device"] == {"0": 10, "1": 100, "2": 50, "3": 10}
        assert all(not i["has_image"] for i in st["images"])
        assert cli.adopt(FakeEngine(), "Ia", 0) is False                       # nothing deposited yet
        cli.deposit(e, "Ia", 0, tier=1)
        e2 = FakeEngine()
        assert cli.adopt(e2, "Ia", 0) is True and e2.attached == 100 * MiB and e2.adopted == (b"DESC\x01", ("weights",))
        n_before = len(FakeBuffer.made)
        assert cli.park(FakeEngine(), "Ia", 0, 80 * MiB)["device"] == 1 and len(FakeBuffer.made) == n_before    # large enough: re-used ...
        assert cli.adopt(FakeEngine(), "Ia", 0) is False                                                        # ... and its old image is void
        assert cli.park(FakeEngine(), "Ia", 0, 300 * MiB, avoid=[0])["bytes"] == 300 * MiB and len(FakeBuffer.made) == n_before + 1
        assert cli.release("Ia") == 1 and cli.release("nobody") == 0
        assert cli.stats()["parked_mib_per_device"]["1"] == 0
        rep, fd = cli._rpc({"op": "bogus"})
        assert rep["ok"] is False and fd is None
        rep, _ = cli._rpc({"op": "park", "instance": "Ie", "bytes": 1, "avoid": [0, 1, 2, 3]})
        assert rep["ok"] is False and "no GPU" in rep["error"]
        # the least-loaded GPU is full (an awake instance owns its HBM): the next candidate takes the buffer; when every candidate is
        # full the park is refused with a reason (the allocator shim then sleeps to the host tier) and nothing is left behind
        FakeBuffer.full = {1}
        assert cli.park(FakeEngine(), "If", 0, 20 * MiB, avoid=[0])["device"] == 3     # loads: 1 -> 0 (full), 3 -> 10, 2 -> 50
        FakeBuffer.full = {1, 2, 3}
        before = cli.stats()
        rep, fd = cli._rpc({"op": "park", "instance": "Ig", "bytes": 20 * MiB, "avoid": [0]})
        assert rep["ok"] is False and fd is None and "no GPU can take 20 MiB" in rep["error"] and "out of memory" in rep["error"]
        assert cli.stats() == before
        FakeBuffer.full = set()
    finally:
        svc.close()
    assert all(b.closed for b in FakeBuffer.made)
