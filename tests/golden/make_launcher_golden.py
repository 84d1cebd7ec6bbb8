"""Writes tests/golden/launcher_rest.json: what the UNMODIFIED reference launcher (inference_server/launcher/launcher.py of
llm-d fast-model-actuation) answers to the request scripts of tests/test_node_agent_differential.py and
tests/test_config0_launcher_plumbing.py.  The node agent is checked against these answers.  Runs on CPU (--mock-gpus, the
children are the config-0 stand-in), from a checkout of that project:

    python tests/golden/make_launcher_golden.py <checkout>/inference_server/launcher/launcher.py
"""
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests import test_config0_launcher_plumbing as C0  # noqa: E402
from tests import test_node_agent_differential as D  # noqa: E402

launcher = os.path.abspath(sys.argv[1])
out = {"generator": "tests/golden/make_launcher_golden.py"}
with tempfile.TemporaryDirectory() as tmp:
    for key, script in (("rest_contract", lambda svc: D._script(svc, D._port())), ("watch", D._watch_script),
                        ("child_dies", D._child_dies_script)):
        svc = D.Service(launcher, tmp)
        try:
            out[key] = D._as_stored(script(svc))
        finally:
            svc.close()
    proc, lport = C0._run_launcher(launcher, os.path.join(tmp, "config0.log"))
    try:
        out["config0"] = C0._controller_sequence(lport, C0._port())
    finally:
        C0._stop(proc)
p = os.path.join(ROOT, "tests", "golden", "launcher_rest.json")
with open(p, "w") as f:
    json.dump(out, f, indent=1)
    f.write("\n")
print("wrote", p)
