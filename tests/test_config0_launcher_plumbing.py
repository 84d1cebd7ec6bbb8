"""BASELINE config 0 (plumbing, no GPU): a launcher creates an instance from the same JSON the Go controller sends
(pkg/controller/dual-pods/launcherclient.go:72-78), forks the child, and the controller's sleep -> is_sleeping -> wake_up
sequence works against the child's port.  The launcher here is the node agent, and every answer must equal what the
UNMODIFIED reference launcher answered to the same sequence (tests/golden/launcher_rest.json, written by
tests/golden/make_launcher_golden.py).  The child is the route-compatible stand-in of SURVEY.md §8c-iv (CPU-worker
semantics: nothing moves)."""
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
AGENT = os.path.join(ROOT, "scripts", "run_node_agent.py")
GOLDEN = os.path.join(ROOT, "tests", "golden", "launcher_rest.json")


def _port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _http(method, url, body=None, timeout=10):
    data = json.dumps(body).encode() if body is not None else (b"" if method in ("POST", "PUT") else None)
    req = urllib.request.Request(url, data=data, method=method, headers={"Content-Type": "application/json"})
    try:
        with urllib.request.urlopen(req, timeout=timeout) as r:
            return r.status, r.read().decode()
    except urllib.error.HTTPError as e:
        return e.code, e.read().decode()


def _wait(url, seconds):
    t0 = time.time()
    while time.time() - t0 < seconds:
        try:
            if _http("GET", url, timeout=2)[0] == 200:
                return True
        except Exception:
            pass
        time.sleep(0.3)
    return False


def _controller_sequence(lport, vport):
    """The controller's calls; returns [route, status, JSON answer] for each, with the child's port written as <port>."""
    obs = []

    def call(label, method, url, body=None):
        st, txt = _http(method, url, body)
        obs.append([label, st, json.loads(txt.replace(str(vport), "<port>")) if txt.startswith("{") else None])
        return st, txt

    body = {"options": f"--model facebook/opt-125m --enable-sleep-mode --port {vport} --host 127.0.0.1",
            "env_vars": {"VLLM_SERVER_DEV_MODE": "1"}, "annotations": {"isc-name": "cfg0", "inference-port": str(vport)}}
    st, txt = call("create", "PUT", f"http://127.0.0.1:{lport}/v2/vllm/instances/cfg0", body)
    assert st == 201, txt
    assert json.loads(txt)["instance_id"] == "cfg0"
    assert call("create-dup", "PUT", f"http://127.0.0.1:{lport}/v2/vllm/instances/cfg0", body)[0] == 409          # duplicate id
    assert _wait(f"http://127.0.0.1:{vport}/health", 60)
    st, txt = call("list", "GET", f"http://127.0.0.1:{lport}/v2/vllm/instances")
    listing = json.loads(txt)
    assert listing["running_instances"] == 1 and listing["instances"][0]["status"] == "running"
    base = f"http://127.0.0.1:{vport}"
    assert json.loads(call("is_sleeping", "GET", base + "/is_sleeping")[1]) == {"is_sleeping": False}
    assert call("sleep", "POST", base + "/sleep")[0] == 200                                                   # ensureUnbound
    assert json.loads(call("is_sleeping", "GET", base + "/is_sleeping")[1]) == {"is_sleeping": True}          # querySleeping
    assert 200 <= call("wake_up", "POST", base + "/wake_up")[0] < 300                                         # wakeSleeper
    assert 200 <= call("wake_up", "POST", base + "/wake_up")[0] < 300                                         # retried: harmless
    assert json.loads(call("is_sleeping", "GET", base + "/is_sleeping")[1]) == {"is_sleeping": False}
    assert call("delete", "DELETE", f"http://127.0.0.1:{lport}/v2/vllm/instances/cfg0")[0] == 200
    assert call("delete", "DELETE", f"http://127.0.0.1:{lport}/v2/vllm/instances/cfg0")[0] == 404
    return obs


def _run_launcher(script, log_path):
    """Start a launcher-compatible service on a free port; returns (process, port)."""
    lport = _port()
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "scripts", "vllm_cpu_standin"), os.path.join(ROOT, "scripts", "k8s_stub"),
                                         ROOT, env.get("PYTHONPATH", "")])
    log = open(log_path, "w")
    proc = subprocess.Popen([sys.executable, script, "--mock-gpus", "--mock-gpu-count", "1", "--host", "127.0.0.1", "--port", str(lport)],
                            env=env, cwd=os.path.dirname(script), stdout=log, stderr=subprocess.STDOUT)
    if not _wait(f"http://127.0.0.1:{lport}/health", 60):
        proc.kill()
        raise AssertionError(open(log_path).read()[-2000:])
    return proc, lport


def _stop(proc):
    proc.terminate()
    try:
        proc.wait(timeout=20)
    except Exception:
        proc.kill()


def test_unmodified_launcher_drives_sleep_wake(built, tmp_path):
    proc, lport = _run_launcher(AGENT, tmp_path / "launcher.log")
    try:
        got = _controller_sequence(lport, _port())
    finally:
        _stop(proc)
    with open(GOLDEN) as f:
        want = json.load(f)["config0"]
    assert [o[0] for o in got] == [o[0] for o in want]
    for g, w in zip(got, want):
        assert g == w, f"{g[0]}: reference {w[1:]} != agent {g[1:]}"
