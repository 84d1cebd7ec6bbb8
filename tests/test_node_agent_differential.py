"""Differential test of the node agent against the UNMODIFIED reference launcher: the same request script runs on CPU
(children = the config-0 stand-in) and every status code, header of interest and JSON shape must agree with what the
reference launcher answered to it (tests/golden/launcher_rest.json, written by tests/golden/make_launcher_golden.py).
Then the node-scoped routes the reference does not have (sleep / wake_up / is_sleeping proxies, swap, sleepers) are
exercised on the agent."""
import json
import os
import socket
import subprocess
import sys
import time
import urllib.error
import urllib.request

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "launcher_rest.json")
AGENT = os.path.join(ROOT, "scripts", "run_node_agent.py")
ENV_PATH = os.pathsep.join([os.path.join(ROOT, "scripts", "vllm_cpu_standin"), os.path.join(ROOT, "scripts", "k8s_stub"), ROOT])


def _port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _http(method, url, body=None, headers=None, timeout=15):
    data = json.dumps(body).encode() if body is not None else (b"" if method in ("POST", "PUT") else None)
    h = {"Content-Type": "application/json"}
    h.update(headers or {})
    req = urllib.request.Request(url, data=data, method=method, headers=h)
    try:
        with urllib.request.urlopen(req, timeout=timeout) as r:
            return r.status, r.read(), {k.lower(): v for k, v in r.headers.items()}
    except urllib.error.HTTPError as e:
        return e.code, e.read(), {k.lower(): v for k, v in e.headers.items()}


def _wait(url, seconds=60):
    t0 = time.time()
    while time.time() - t0 < seconds:
        try:
            if _http("GET", url, timeout=2)[0] == 200:
                return True
        except Exception:
            pass
        time.sleep(0.2)
    return False


class Service:
    """A launcher-compatible REST service (the node agent, or the reference launcher when the golden file is written)."""

    def __init__(self, script, log_dir):
        self.port = _port()
        env = dict(os.environ)
        env["PYTHONPATH"] = os.pathsep.join([ENV_PATH, env.get("PYTHONPATH", "")])
        log = os.path.join(log_dir, "service.log")
        self.log = open(log, "w")
        self.proc = subprocess.Popen([sys.executable, script, "--mock-gpus", "--host", "127.0.0.1", "--port", str(self.port)],
                                     env=env, cwd=os.path.dirname(script), stdout=self.log, stderr=subprocess.STDOUT)
        self.base = f"http://127.0.0.1:{self.port}"
        assert _wait(self.base + "/health"), open(log).read()[-2000:]

    def close(self):
        self.proc.terminate()
        try:
            self.proc.wait(timeout=30)
        except Exception:
            self.proc.kill()


@pytest.fixture()
def mine(built, tmp_path):
    svc = Service(AGENT, str(tmp_path))
    yield svc
    svc.close()


def _reference(key):
    """What the reference launcher answered to the same script (JSON: tuples are stored as lists)."""
    with open(GOLDEN) as f:
        return json.load(f)[key]


def _as_stored(x):
    return json.loads(json.dumps(x))


def _shape(x):
    """Structure of a JSON value with volatile leaves (ids, revisions, pids, free text) reduced to their types."""
    if isinstance(x, dict):
        return {k: _shape(v) for k, v in sorted(x.items())}
    if isinstance(x, list):
        return [_shape(v) for v in x]
    return type(x).__name__


def _script(svc, vport):
    """One pass of the launcher REST contract; returns a list of comparable observations."""
    obs = []
    b = svc.base

    def rec(label, st, body, headers=None, keep=()):
        try:
            j = json.loads(body) if body else None
        except Exception:
            j = None
        obs.append((label, st, _shape(j), {k: (headers or {}).get(k) for k in keep}))
        return j

    cfg = {"options": f"--model facebook/opt-125m --enable-sleep-mode --port {vport} --host 127.0.0.1",
           "env_vars": {"VLLM_SERVER_DEV_MODE": "1"}, "annotations": {"isc-name": "d", "inference-port": str(vport)}, "gpu_uuids": ["GPU-0"]}
    rec("health", *_http("GET", b + "/health")[:2])
    j = rec("list-empty", *_http("GET", b + "/v2/vllm/instances")[:2])
    assert j["total_instances"] == 0 and j["revision"] == 0
    j = rec("put", *_http("PUT", b + "/v2/vllm/instances/inst-a", cfg)[:2])
    assert j["instance_id"] == "inst-a" and j["status"] == "running" and j["revision"] == 1
    assert j["env_vars"]["CUDA_VISIBLE_DEVICES"] == "0"                      # GPU-0 -> index 0 (mock translator)
    rec("put-dup", *_http("PUT", b + "/v2/vllm/instances/inst-a", cfg)[:2])
    rec("put-bad-body", *_http("PUT", b + "/v2/vllm/instances/inst-x", {"nope": 1})[:2])
    assert _wait(f"http://127.0.0.1:{vport}/health")
    j = rec("get", *_http("GET", b + "/v2/vllm/instances/inst-a")[:2])
    rec("get-404", *_http("GET", b + "/v2/vllm/instances/missing")[:2])
    j = rec("list", *_http("GET", b + "/v2/vllm/instances")[:2])
    assert j["running_instances"] == 1
    j = rec("list-ids", *_http("GET", b + "/v2/vllm/instances?detail=false")[:2])
    assert j["instance_ids"] == ["inst-a"] and j["count"] == 1
    # the child writes its log through the redirected stdout/stderr: wait for some bytes
    t0 = time.time()
    while time.time() - t0 < 20:
        st, body, h = _http("GET", b + "/v2/vllm/instances/inst-a/log")
        if st == 200 and len(body) > 40:
            break
        time.sleep(0.3)
    total = int(h["content-range"].split("/")[1])
    obs.append(("log-full", st, h["content-range"].startswith("bytes 0-"), h.get("accept-ranges")))
    st, part, h = _http("GET", b + "/v2/vllm/instances/inst-a/log", headers={"Range": "bytes=5-14"})
    obs.append(("log-206", st, len(part), h["content-range"].split("/")[0]))
    assert part == body[5:15]
    st, tail, h = _http("GET", b + "/v2/vllm/instances/inst-a/log", headers={"Range": "bytes=10-"})
    obs.append(("log-open-range", st, h["content-range"].startswith("bytes 10-")))
    st, _, h = _http("GET", b + "/v2/vllm/instances/inst-a/log", headers={"Range": f"bytes={total + 1000}-"})
    obs.append(("log-416", st, h["content-range"].startswith("bytes */")))
    obs.append(("log-400", _http("GET", b + "/v2/vllm/instances/inst-a/log", headers={"Range": "bytes=9-3"})[0]))
    obs.append(("log-400b", _http("GET", b + "/v2/vllm/instances/inst-a/log", headers={"Range": "lines=1-2"})[0]))
    obs.append(("log-404", _http("GET", b + "/v2/vllm/instances/missing/log")[0]))
    obs.append(("watch-410", _http("GET", b + "/v2/vllm/instances/watch?since=-5")[0]))
    j = rec("post-generated", *_http("POST", b + "/v2/vllm/instances", {"options": f"--port {_port()} --host 127.0.0.1"})[:2])
    gen_id = j["instance_id"]
    assert len(gen_id) == 36                                                 # uuid4
    j = rec("delete", *_http("DELETE", b + f"/v2/vllm/instances/{gen_id}")[:2])
    assert j["status"] == "stopped"
    rec("delete-404", *_http("DELETE", b + f"/v2/vllm/instances/{gen_id}")[:2])
    j = rec("delete-all", *_http("DELETE", b + "/v2/vllm/instances")[:2])
    assert j["total_stopped"] == 1 and j["status"] == "all_stopped"
    j = rec("list-after", *_http("GET", b + "/v2/vllm/instances")[:2])
    assert j["total_instances"] == 0 and j["revision"] == 4                 # created, created, deleted, deleted
    return obs


def test_same_rest_contract_as_the_reference_launcher(mine):
    a = _reference("rest_contract")
    b = _as_stored(_script(mine, _port()))
    assert [x[0] for x in a] == [x[0] for x in b]
    for ra, rb in zip(a, b):
        assert ra == rb, f"{ra[0]}: reference {ra[1:]} != agent {rb[1:]}"


def _read_events(url, n, timeout=20):
    out = []
    with urllib.request.urlopen(url, timeout=timeout) as r:
        while len(out) < n:
            line = r.readline()
            if not line:
                break
            out.append(json.loads(line))
    return out


def _watch_script(svc):
    vport = _port()
    cfg = {"options": f"--port {vport} --host 127.0.0.1", "annotations": {"inference-port": str(vport)}}
    assert _http("PUT", svc.base + "/v2/vllm/instances/w1", cfg)[0] == 201
    import threading

    got = []
    t = threading.Thread(target=lambda: got.extend(_read_events(svc.base + "/v2/vllm/instances/watch", 3)))
    t.start(); time.sleep(1.0)                                           # watcher connected: gets CREATED(w1) first
    assert _http("PUT", svc.base + "/v2/vllm/instances/w2", {"options": f"--port {_port()} --host 127.0.0.1"})[0] == 201
    assert _http("DELETE", svc.base + "/v2/vllm/instances/w2")[0] == 200
    t.join(timeout=30)
    seq = [(e["type"], e["object"]["instance_id"], e["object"]["status"], sorted(e["object"])) for e in got]
    # resume from revision 1: only what happened after the first create
    later = _read_events(svc.base + "/v2/vllm/instances/watch?since=1", 2)
    seq.append([(e["type"], e["object"]["instance_id"], e["object"]["revision"]) for e in later])
    _http("DELETE", svc.base + "/v2/vllm/instances")
    return seq


def test_watch_stream_matches_the_reference(mine):
    seq = _as_stored(_watch_script(mine))
    assert _reference("watch") == seq
    assert [e[0] for e in seq[:3]] == ["CREATED", "CREATED", "DELETED"]


def _child_dies_script(svc):
    vport = _port()
    assert _http("PUT", svc.base + "/v2/vllm/instances/dies", {"options": f"--port {vport} --host 127.0.0.1"})[0] == 201
    assert _wait(f"http://127.0.0.1:{vport}/health")
    psutil = pytest.importorskip("psutil")
    pid = next((c.pid for c in psutil.net_connections(kind="tcp") if c.laddr and c.laddr.port == vport and c.status == "LISTEN" and c.pid), None)
    if pid is None:
        pytest.skip("cannot find the child's pid")
    os.kill(pid, 9)
    ev = _read_events(svc.base + "/v2/vllm/instances/watch?since=1", 1)
    st = json.loads(_http("GET", svc.base + "/v2/vllm/instances/dies")[1])
    _http("DELETE", svc.base + "/v2/vllm/instances")
    return (ev[0]["type"], ev[0]["object"]["status"], ev[0]["object"]["exit_code"], st["status"], sorted(ev[0]["object"]))


def test_stopped_event_when_a_child_dies(mine):
    """A child that exits by itself is reported as STOPPED with its exit code, and stays listed as 'stopped'."""
    ref, mine = _reference("child_dies"), _as_stored(_child_dies_script(mine))
    assert mine[:4] == ["STOPPED", "stopped", -9, "stopped"]
    # same event type, same keys, same final listing.  The reference's event body is racy here: its exit watcher fires
    # when the child's sentinel pipe closes, which the kernel does BEFORE the process becomes reapable, so
    # `is_alive()`/`exitcode` inside the callback can still say running/None (launcher.py:256-266,372-382).
    assert ref[0] == mine[0] and ref[3] == mine[3] and ref[4] == mine[4]
    assert (ref[1], ref[2]) in {("stopped", -9), ("running", None)}


def test_node_scoped_actuation_routes(mine):
    pa, pb = _port(), _port()
    for iid, p in (("model-a", pa), ("model-b", pb)):
        cfg = {"options": f"--enable-sleep-mode --port {p} --host 127.0.0.1", "env_vars": {"VLLM_SERVER_DEV_MODE": "1"},
               "annotations": {"inference-port": str(p)}, "gpu_uuids": ["GPU-3"]}
        assert _http("PUT", mine.base + f"/v2/vllm/instances/{iid}", cfg)[0] == 201
    assert _wait(f"http://127.0.0.1:{pa}/health") and _wait(f"http://127.0.0.1:{pb}/health")
    j = json.loads(_http("POST", mine.base + "/v2/vllm/instances/model-b/sleep")[1])
    assert j["status_code"] == 200 and j["action"] == "sleep" and j["seconds"] >= 0
    assert json.loads(_http("GET", mine.base + "/v2/vllm/instances/model-b/is_sleeping")[1])["is_sleeping"] is True
    assert json.loads(_http("GET", f"http://127.0.0.1:{pb}/is_sleeping")[1]) == {"is_sleeping": True}   # really reached the instance
    st, body, _ = _http("POST", mine.base + "/v2/node/swap", {"sleep": "model-a", "wake": "model-b"})    # sleep(A) || wake(B)
    j = json.loads(body)
    assert st == 200 and j["sleep"]["status_code"] == 200 and j["wake"]["status_code"] == 200
    assert json.loads(_http("GET", f"http://127.0.0.1:{pa}/is_sleeping")[1]) == {"is_sleeping": True}
    assert json.loads(_http("GET", f"http://127.0.0.1:{pb}/is_sleeping")[1]) == {"is_sleeping": False}
    s = json.loads(_http("GET", mine.base + "/v2/node/sleepers")[1])
    assert s["sleeping_count"] == 1 and {x["instance_id"]: x["is_sleeping"] for x in s["sleepers"]} == {"model-a": True, "model-b": False}
    assert all(x["cuda_visible_devices"] == "3" for x in s["sleepers"])
    assert _http("POST", mine.base + "/v2/node/swap", {"sleep": "nope", "wake": "model-b"})[0] == 404
    assert _http("POST", mine.base + "/v2/vllm/instances/nope/wake_up")[0] == 404
    assert json.loads(_http("POST", mine.base + "/v2/vllm/instances/model-a/wake_up")[1])["status_code"] == 200
