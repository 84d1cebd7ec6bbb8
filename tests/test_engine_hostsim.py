"""The engine's HOST logic on CPU.  The host translation units (csrc/fma_engine.cu, fma_sleep.cu, fma_wake.cu, fma_load.cu,
fma_image.cu) are compiled with g++ against a host simulation of the CUDA runtime +
VMM driver calls (tests/cpp/hostsim/, test infrastructure: mmap-backed VMM with the real map/unmap semantics, eager
streams) and host stand-ins for the kernel launch wrappers, then

  1. the GPU parity suite (tests/test_gpu_parity.py, everything that does not need torch on a GPU) runs against that
     library in a subprocess — segment table, arenas, runs, ring, mapper/unmapper threads, modes, tiers incl. the
     peer tier, swap, cold load, error handling;
  2. a C++ scenario drives the C-ABI under ThreadSanitizer and under AddressSanitizer+UBSan+LeakSanitizer, including
     a failed wake (injected cuMemCreate failure) followed by the controller's retry, and checks that destroying the
     engines leaves no mapping and no handle behind.

The product library contains none of this: without a GPU it refuses to run (tests/test_abi.py)."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIM = os.path.join(ROOT, "tests", "cpp", "hostsim")
CSRC = os.path.join(ROOT, "llm-d-fast-model-actuation_b200", "csrc")
INC = ["-I/usr/local/cuda/include", "-I" + CSRC, "-I" + os.path.join(ROOT, "include")]
HOST_TUS = ["fma_engine.cu", "fma_sleep.cu", "fma_wake.cu", "fma_load.cu", "fma_image.cu", "fma_gate.cu", "fma_pull.cu"]   # the host engine (no kernels): csrc/Makefile HOST_SRCS
SRCS = ["-x", "c++", *[os.path.join(CSRC, f) for f in HOST_TUS], os.path.join(SIM, "hostsim_cuda.cpp"), os.path.join(SIM, "hostsim_kernels.cpp")]


def _have_cuda_headers():
    return os.path.exists("/usr/local/cuda/include/cuda_runtime.h")


@pytest.fixture(scope="module")
def hostsim_lib(tmp_path_factory):
    if not _have_cuda_headers():
        pytest.skip("CUDA headers not installed")
    out = str(tmp_path_factory.mktemp("hostsim") / "libfma_b200_hostsim.so")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-g", "-shared", "-fPIC", "-fvisibility=hidden", *INC, *SRCS, "-o", out, "-lpthread"])
    return out


def _xdist():
    """The ~100 simulated GPU tests are independent (an engine each): spread them over a few workers when pytest-xdist is there."""
    try:
        import xdist  # noqa: F401
    except ImportError:
        return []
    return ["-n", str(max(1, min(4, (os.cpu_count() or 2) // 2)))]


def test_parity_suite_against_the_host_simulated_engine(hostsim_lib, oracle):
    env = dict(os.environ, FMA_B200_LIB=hostsim_lib, FMA_HOSTSIM="1", HOSTSIM_DEVICES="2")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(ROOT, "tests", "test_gpu_parity.py"), os.path.join(ROOT, "tests", "test_gpu_http.py"), "-x", "-q", "-m", "gpu",
                        "-k", "not shim and not torch_pool and not full_size", "-p", "no:cacheprovider", *_xdist()],
                       env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0, tail
    assert " passed" in r.stdout and "failed" not in r.stdout and " error" not in r.stdout.lower(), tail


def test_engine_scenario_under_sanitizers(tmp_path):
    """ThreadSanitizer and ASan+UBSan+LeakSan builds of the same scenario, compiled and run side by side."""
    if not _have_cuda_headers():
        pytest.skip("CUDA headers not installed")
    from concurrent.futures import ThreadPoolExecutor

    def one(san, flags):
        exe = str(tmp_path / f"engine_{san}")
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-g", *flags, *INC, *SRCS, os.path.join(SIM, "engine_sanitizer_test.cpp"),
                               "-o", exe, "-lpthread"])
        env = dict(os.environ, ASAN_OPTIONS="detect_leaks=1", TSAN_OPTIONS="halt_on_error=1", HOSTSIM_DEVICES="2")
        r = subprocess.run([exe], env=env, capture_output=True, text=True, timeout=900)
        return san, r.returncode, r.stdout + r.stderr

    with ThreadPoolExecutor(2) as pool:
        results = list(pool.map(lambda a: one(*a), [("tsan", ["-fsanitize=thread"]), ("asan", ["-fsanitize=address,undefined", "-fno-omit-frame-pointer"])]))
    for san, rc, out in results:
        assert rc == 0 and "engine sanitizer scenario ok" in out, (san, out[-3000:])
        assert "WARNING: ThreadSanitizer" not in out and "ERROR: AddressSanitizer" not in out and "runtime error:" not in out, (san, out[-3000:])


def test_bench_packed_image_child_runs_against_the_host_simulated_engine(hostsim_lib, oracle):
    """bench.py's packed-image extra (its own process at N=1): fill with bf16 dummy weights, sleep/wake with config.pack,
    digests before == after, 0.758 of the bytes stored.  torch is replaced by tests/stubs/torch (numpy)."""
    import json

    env = dict(os.environ, FMA_B200_LIB=hostsim_lib, FMA_HOSTSIM="1", HOSTSIM_DEVICES="1",
               PYTHONPATH=os.path.join(ROOT, "tests", "stubs") + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--packed-child", "--workload", "tiny-llama-test",
                        "--kv-gib", "0.03125", "--steps", "2", "--warmup", "1"], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["bit_exact"] is True and out["image_packed"] is True
    assert 0.75 < out["stored_frac"] < 0.80 and out["e2e_effective_gbs"] > out["e2e_link_gbs"] > 0
    inc = out["incremental_sleep"]
    assert inc["bit_exact"] is True and inc["sleep_bytes_copied"][0] > 0 and inc["sleep_bytes_copied"][1:] == [0, 0, 0]


def test_vllm_loader_streaming_core_against_the_host_simulated_engine(hostsim_lib, tmp_path):
    """stream_tensors(): two safetensors files, small windows, a staging segment that grows, views that alias it, and a
    drain() before every reuse — every tensor arrives with the file's bytes, in file order."""
    code = r"""
import ctypes, json, os, sys
import numpy as np
sys.path.insert(0, %r)
import fma_b200
from fma_b200 import loader, vllm_loader
rng = np.random.default_rng(3)
files, want = [], {}
for f in range(2):
    tensors = []
    for i, n in enumerate([1000, 70000, 3 << 20, 12, 0, 5 << 20, 4096]):
        name = f"f{f}.t{i}"
        raw = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        tensors.append((name, "U8", (n,), raw)); want[name] = raw
    path = os.path.join(%r, f"m-{f}.safetensors")
    loader.write_safetensors(path, tensors); files.append(path)
eng = fma_b200.Engine(0)
drains, live = [0], []
def view(ptr, off, t):
    return (ptr + off, t.nbytes)
def drain():
    drains[0] += 1
stats = {}
got = {}
for name, (addr, n) in vllm_loader.stream_tensors(eng, files, view, drain=drain, window_bytes=4 << 20, stats=stats):
    got[name] = ctypes.string_at(addr, n)            # host simulation: device memory is host memory; consume before the next window
assert list(got) == [k for k in want if len(want[k])], list(got)
assert all(got[k] == want[k] for k in got)
assert stats["windows"] >= 4 and drains[0] == stats["windows"] + 1 and stats["bytes"] >= sum(len(v) for v in want.values())
assert eng.segment_count() == 0                      # the staging segment is gone
print("ok")
""" % (ROOT, str(tmp_path))
    env = dict(os.environ, FMA_B200_LIB=hostsim_lib, FMA_HOSTSIM="1", HOSTSIM_DEVICES="1")
    r = subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, (r.stdout + r.stderr)[-3000:]


def test_bench_main_flow_runs_against_the_host_simulated_engine(hostsim_lib, oracle, tmp_path):
    """The whole of bench.py's own arm at N=1 — table, fill, digests, timed cycles, JSON line with every contract key,
    cpu_baseline fallback (the oracle port: vLLM's allocator cannot load here) and the packed_image child — with torch
    replaced by tests/stubs/torch.  Numbers are meaningless here; the flow and the keys are what is checked.  --dump-outputs
    writes the restored weights (digests == the oracle's, a byte sample), and a second run with the same arguments writes the
    same arrays."""
    import json

    import numpy as np

    env = dict(os.environ, FMA_B200_LIB=hostsim_lib, FMA_HOSTSIM="1", HOSTSIM_DEVICES="2",
               PYTHONPATH=os.path.join(ROOT, "tests", "stubs") + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny-llama-test", "--kv-gib", "0.03125",
                        "--steps", "2", "--warmup", "3", "--swap-models", "tiny-llama-test,tiny-llama-test", "--scaling-workload", "opt-125m",
                        "--extras-kv-gib", "0.03125", "--timeline", str(tmp_path / "tl"), "--dump-outputs", str(tmp_path / "out")],
                       env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["steps"] == 2 and len(out["wake_latency_s_steps"]) == 2
    r2 = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny-llama-test", "--kv-gib", "0.03125",
                         "--steps", "1", "--warmup", "3", "--extras", "", "--packed-extra", "0", "--no-cpu-baseline",
                         "--dump-outputs", str(tmp_path / "out2")], env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r2.returncode == 0, (r2.stdout + r2.stderr)[-3000:]
    assert json.loads(r2.stdout.strip().splitlines()[-1])["steps"] == 1
    import fma_b200  # noqa: F401
    from fma_b200 import workloads as W

    weights = [s for s in W.allocation_table("tiny-llama-test") if s.tag == "weights"]
    want, first = [], 0
    for s in weights:
        want.append(oracle.digest(oracle.fill(s.bytes, 1234, first)))
        first += s.bytes // 8
    for name in ("weights_digest", "weights_sample"):
        a, b = np.load(tmp_path / "out" / f"{name}.npy"), np.load(tmp_path / "out2" / f"{name}.npy")
        assert a.dtype in (np.float32, np.float64) and a.nbytes <= 64 << 20 and np.array_equal(a, b), name
    dg = np.load(tmp_path / "out" / "weights_digest.npy")
    assert [int(hi) << 32 | int(lo) for hi, lo in dg] == want
    sample = np.load(tmp_path / "out" / "weights_sample.npy")
    assert sample.shape == (2048, 4096) and sample.min() >= 0 and sample.max() <= 255 and sample.std() > 50
    assert out["swap_config4"].get("bit_exact") is True and out["swap_config4"]["cycles"] == 20, out["swap_config4"]
    assert out["n1_on_scaling_workload"].get("bit_exact") is True, out["n1_on_scaling_workload"]
    assert out["multipath_wake"].get("bit_exact") is True and out["multipath_wake"]["rows"][0]["paths"] == 2, out["multipath_wake"]
    assert out["config"]["segments_per_rank"] > 0 and "phases" in out["config"]
    assert out["wake_latency_s_min_max"][0] <= out["wake_latency_s"] <= out["wake_latency_s_min_max"][1]
    tl = open(tmp_path / "tl" / "n1_rank0.csv").read()
    assert "wake,map_backed" in tl and "wake,total" in tl and "sleep,unmap" in tl and "wake,kernel" in tl, tl[:600]
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                "data", "config", "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks", "packed_image"):
        assert key in out, key
    assert out["bit_exact"] is True and out["n_gpus"] == 1 and out["gpu_launches"] > 0
    assert out["e2e"]["link_bytes_per_step"] == out["e2e"]["h2d_bytes_per_step"]          # not packed: every weight byte crosses the link
    assert out["cpu_baseline"]["kind"] == "port"
    assert out["packed_image"].get("bit_exact") is True and out["packed_image"]["image_packed"] is True


def test_smoke_entry_point_runs_against_the_host_simulated_engine(hostsim_lib, oracle):
    """__graft_entry__.smoke() — what the driver runs on cuda:0 — with the host-simulated engine: its checks (digests, packed
    host image == oracle gather, addresses, bytes) hold in all three modes."""
    env = dict(os.environ, FMA_B200_LIB=hostsim_lib, FMA_HOSTSIM="1", HOSTSIM_DEVICES="1")
    r = subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.smoke()"], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "smoke ok" in r.stdout, (r.stdout + r.stderr)[-3000:]


@pytest.mark.parametrize("build", ["linked", "tsan"])
def test_native_server_speaks_the_controller_contract_over_the_host_simulated_engine(hostsim_lib, tmp_path, build):
    """csrc/fma_served.cpp — the compiled host side: the reference's cmd/test-server (main.go:56-91) with the atomic bool
    replaced by engines.  Built against the host-simulated library, two ranks; the controller's sequence, idempotence and
    retries, level / tag-selective wake, wrong methods, and bit-identity of the weights (K3 digests) across sleep -> wake."""
    import json
    import time
    import urllib.error
    import urllib.request

    exe = str(tmp_path / "fma_served")
    libdir = os.path.dirname(hostsim_lib)
    if build == "linked":      # against the shared library, as the product binary is
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-g", "-Wall", "-Wextra", os.path.join(CSRC, "fma_served.cpp"), "-o", exe,
                               "-L" + libdir, "-l:" + os.path.basename(hostsim_lib), "-Wl,-rpath," + libdir, "-lpthread"])
    else:                      # server + engine + simulation in one ThreadSanitizer build: connection threads vs rank threads vs engine threads
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-g", "-fsanitize=thread", *INC, *SRCS, os.path.join(CSRC, "fma_served.cpp"), "-o", exe, "-lpthread"])
    env = dict(os.environ, HOSTSIM_DEVICES="2", TSAN_OPTIONS="halt_on_error=1")
    p = subprocess.Popen([exe, "--port", "0", "--device", "0", "--device", "1", "--seg", "weights:6", "--seg", "weights:2", "--seg", "kv_cache:8",
                          "--seg", "weights:4"], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    try:
        line = p.stdout.readline()
        assert line.startswith("listening on "), line + p.stderr.read()
        base = f"http://127.0.0.1:{int(line.split()[-1])}"

        def call(method, path):
            req = urllib.request.Request(base + path, data=b"" if method == "POST" else None, method=method, headers={"Content-Type": "application/json"})
            try:
                with urllib.request.urlopen(req, timeout=60) as r:
                    return r.status, r.read()
            except urllib.error.HTTPError as e:
                return e.code, e.read()

        assert call("GET", "/health") == (200, b"OK\n")
        assert json.loads(call("GET", "/is_sleeping")[1]) == {"is_sleeping": False}
        st, before = call("GET", "/digests")
        assert st == 200 and len(json.loads(before)) == 2 and len(json.loads(before)[0]) == 3
        # the controller's sequence (inference-server.go:1329-1339, 1595-1607, 1118-1137)
        assert call("POST", "/sleep") == (200, b"")
        assert json.loads(call("GET", "/is_sleeping")[1]) == {"is_sleeping": True}
        assert call("GET", "/digests")[0] == 409
        stats = json.loads(call("GET", "/stats")[1])
        assert [r["sleep_bytes_offloaded"] for r in stats["ranks"]] == [12 << 20] * 2 and all(r["hbm_mapped_bytes"] == 0 for r in stats["ranks"])
        assert call("POST", "/sleep") == (200, b"")                       # twice: harmless
        assert call("POST", "/wake_up") == (200, b"") and call("POST", "/wake_up") == (200, b"")   # retried by the controller
        assert json.loads(call("GET", "/is_sleeping")[1]) == {"is_sleeping": False}
        assert call("GET", "/digests") == (200, before)                   # weights bit-identical on every rank
        # level 2 + tag-selective wake (vLLM API compatibility)
        assert call("POST", "/sleep?level=2&mode=abort")[0] == 200
        assert call("POST", "/wake_up?tags=weights")[0] == 200 and json.loads(call("GET", "/is_sleeping")[1])["is_sleeping"] is True
        assert call("POST", "/wake_up?tags=bogus")[0] == 200 and json.loads(call("GET", "/is_sleeping")[1])["is_sleeping"] is True
        assert call("POST", "/wake_up?tags=kv_cache")[0] == 200 and json.loads(call("GET", "/is_sleeping")[1])["is_sleeping"] is False
        assert json.loads(call("GET", "/stats")[1])["ranks"][0]["wake_bytes_restored"] == 0      # level 2 offloads nothing
        # errors
        assert call("GET", "/sleep")[0] == 405 and call("POST", "/is_sleeping")[0] == 405 and call("GET", "/nope")[0] == 404
        assert call("POST", "/sleep?level=x")[0] == 422
    finally:
        p.terminate()
        try:
            p.wait(timeout=30)
        except subprocess.TimeoutExpired:
            p.kill()
    err = p.stderr.read()
    assert p.returncode == 0 and "WARNING: ThreadSanitizer" not in err, err[-3000:]


_PARKING_INSTANCE = r"""
import os, sys, json
sys.path.insert(0, {root!r})
import fma_b200
from fma_b200 import workloads as W, _lib as L
from fma_b200.parking import ParkingClient
phase, iid = sys.argv[1], sys.argv[2]
eng = fma_b200.Engine(0)
table = W.allocation_table("tiny-llama-test", kv_cache_bytes=32 << 20, kv_tensors=2)
for s in table: eng.alloc(s.bytes, s.tag)
cli = ParkingClient()                                  # FMA_NODE_AGENT_SOCK
Wb = sum(s.bytes for s in table if s.tag == "weights")
if phase == "park":
    first = 0
    for i, s in enumerate(table):
        if s.tag == "weights":
            eng.fill(i, 77, first); first += s.bytes // 8
    print(json.dumps(eng.digest_all(["weights"])), flush=True)
    rep = cli.park(eng, iid, 0, Wb, avoid=[0])
    assert rep["device"] != 0
    eng.sleep(["weights"], tier=L.FMA_TIER_PEER, flags=L.FMA_FLAG_VERIFY)
    cli.deposit(eng, iid, 0)
    os._exit(0)                                        # dies asleep
elif phase == "remote_paths":                          # MULTI-PATH wake across processes through the owner's helpers
    first = 0
    for i, s in enumerate(table):
        if s.tag == "weights":
            eng.fill(i, 79, first); first += s.bytes // 8
    before = eng.digest_all(["weights"])
    assert cli.attach_remote_paths(eng, iid, 0, n_helpers=2, avoid=[0], slot_bytes=4 << 20, slots=3) == 2
    eng.host_reserve(Wb)
    remote = []
    for rnd in range(3):
        eng.sleep(["weights"], flags=L.FMA_FLAG_VERIFY)
        if rnd != 1:
            assert cli.request_pull(eng, iid, 0, timeout_s=20.0) == 2
        eng.wake(None, flags=L.FMA_FLAG_VERIFY)
        assert eng.digest_all(["weights"]) == before
        remote.append(sum(r["bytes"] for r in eng.timeline() if r["kind"] == "path_chunks" and r["idx"] < 0))
    assert remote[0] > 0 and remote[1] == 0 and remote[2] > 0, remote
    print(json.dumps(remote), flush=True)
    cli.release(iid)
    os._exit(0)
elif phase == "park_host":                             # HOST tier: the memfd behind the store goes to the owner
    first = 0
    for i, s in enumerate(table):
        if s.tag == "weights":
            eng.fill(i, 78, first); first += s.bytes // 8
    print(json.dumps(eng.digest_all(["weights"])), flush=True)
    eng.sleep(["weights"], flags=L.FMA_FLAG_VERIFY)
    cli.deposit_host(eng, iid, 0)
    os._exit(0)
elif phase == "adopt_host":
    assert cli.adopt(eng, iid, 0) is False and cli.adopt_host(eng, iid, 0) is True and eng.is_sleeping()
    eng.wake(None, flags=L.FMA_FLAG_VERIFY)
    print(json.dumps(eng.digest_all(["weights"])), flush=True)
else:
    assert cli.adopt(eng, iid, 0) is True and eng.is_sleeping()
    eng.wake(None, flags=L.FMA_FLAG_VERIFY)
    print(json.dumps(eng.digest_all(["weights"])), flush=True)
    assert cli.adopt(fma_b200.Engine(0), "nobody", 0) is False
"""


def test_node_level_parking_service_keeps_a_dead_instances_image(hostsim_lib, tmp_path, sock_dir):
    """fma_b200.parking: the node agent's ParkingService owns exportable parking buffers and serves fds over a unix socket; an
    instance parks its weights there, deposits the descriptor and DIES; a fresh instance with the same ID finds the image, attaches,
    adopts and wakes with identical K3 digests; the owner's accounting (MiB per GPU — what a sleeper budget needs,
    inference-server.go:1609-1636) follows.  Host-simulated engine; the C-ABI underneath is GPU-tested in tests/test_gpu_parity.py."""
    import json

    env = dict(os.environ, FMA_B200_LIB=hostsim_lib, FMA_HOSTSIM="1", HOSTSIM_DEVICES="3", FMA_NODE_AGENT_SOCK=os.path.join(sock_dir, "park.sock"))
    owner = r"""
import os, sys, json, subprocess
sys.path.insert(0, %r)
import fma_b200
from fma_b200.parking import ParkingService, ParkingClient
svc = ParkingService(os.environ["FMA_NODE_AGENT_SOCK"], n_devices=3)
svc.start()
script = sys.argv[1]
a = subprocess.run([sys.executable, script, "park", "Iabci"], capture_output=True, text=True, timeout=300)
assert a.returncode == 0, a.stdout + a.stderr
st = svc.stats()
assert st["images"] == [{"instance": "Iabci", "rank": 0, "device": 1, "mib": st["images"][0]["mib"], "has_image": True}] and st["parked_mib_per_device"]["1"] > 0, st
b = subprocess.run([sys.executable, script, "adopt", "Iabci"], capture_output=True, text=True, timeout=300)
assert b.returncode == 0, b.stdout + b.stderr
assert json.loads(a.stdout.strip().splitlines()[0]) == json.loads(b.stdout.strip().splitlines()[-1])
assert ParkingClient().stats()["ok"] and ParkingClient().release("Iabci") == 1
assert svc.stats()["images"] == [] and svc.stats()["parked_mib_per_device"]["1"] == 0
# the same for the HOST tier: the memfd behind a sleeping instance's store is kept by the owner
env_h = dict(os.environ, FMA_HOST_STORE_SHM="1")
c = subprocess.run([sys.executable, script, "park_host", "Ihosti"], capture_output=True, text=True, timeout=300, env=env_h)
assert c.returncode == 0, c.stdout + c.stderr
assert [h["instance"] for h in svc.stats()["host_images"]] == ["Ihosti"] and svc.stats()["host_images"][0]["mib"] > 0
d = subprocess.run([sys.executable, script, "adopt_host", "Ihosti"], capture_output=True, text=True, timeout=300, env=env_h)
assert d.returncode == 0, d.stdout + d.stderr
assert json.loads(c.stdout.strip().splitlines()[0]) == json.loads(d.stdout.strip().splitlines()[-1])
assert ParkingClient().release("Ihosti") == 1 and svc.stats()["host_images"] == []
# MULTI-PATH wake across processes: the owner's helper GPUs pull for an instance that cannot see them
e = subprocess.run([sys.executable, script, "remote_paths", "Iremotei"], capture_output=True, text=True, timeout=300, env=dict(env_h, FMA_PULL_TIMEOUT_S="20"))
assert e.returncode == 0, e.stdout + e.stderr
svc.close()
print("parking service ok")
""" % ROOT
    script = tmp_path / "instance.py"
    script.write_text(_PARKING_INSTANCE.format(root=ROOT))
    r = subprocess.run([sys.executable, "-c", owner, str(script)], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "parking service ok" in r.stdout, (r.stdout + r.stderr)[-3000:]
