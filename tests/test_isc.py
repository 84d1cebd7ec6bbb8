"""Instance-ID / VllmConfig derivation (SURVEY.md §8f-2; pkg/controller/dual-pods/inference-server.go:801-829).

The marshaller is pinned against the reference's generated CRDs (same sigs.k8s.io/yaml stack, 8834 lines, byte for byte);
the ID composition has no reference vector (no expected ID anywhere in the reference): hand-derived expectations."""
import base64
import hashlib
import importlib

import pytest

isc = importlib.import_module("llm-d-fast-model-actuation_b200.isc")


def test_top_level_keys_are_sorted_and_empty_fields_omitted():
    j = isc.model_server_config_json(8005, "--model m", {"B": "2x", "A": "x"}, None, {})
    assert isc.go_yaml_marshal(j) == b"env_vars:\n  A: x\n  B: 2x\noptions: --model m\nport: 8005\n"
    assert isc.go_yaml_marshal(isc.model_server_config_json(8000)) == b"port: 8000\n"


@pytest.mark.parametrize("text,expected", [
    ("1", '"1"'), ("0.4", '"0.4"'), ("yes", '"yes"'), ("True", '"True"'), ("null", '"null"'), ("~", '"~"'),
    ("0x1F", '"0x1F"'), ("1e3", '"1e3"'), ("1_000", '"1_000"'), ("2024-01-02", '"2024-01-02"'), ("1:30", '"1:30"'),
    (".5", '".5"'), ("-.inf", '"-.inf"'), ("0b101", '"0b101"'), ("+12", '"+12"'),
    # strings that stay plain in yaml.v2 (PyYAML's own resolver would quote "=" and not "1e3")
    ("=", "="), ("x", "x"), ("--port=1", "--port=1"), ("1.2.3", "1.2.3"), ("GPU-0", "GPU-0"), ("nope", "nope"),
    ("0x", "0x"), ("12ab", "12ab"), ("-", "'-'"), ("2024-13-02", "2024-13-02"),
    # not plain-able: the emitter picks single quotes, then double quotes
    ("a: b", "'a: b'"), ("a #b", "'a #b'"), (" lead", "' lead'"), ("trail ", "'trail '"), ("it's: x", "'it''s: x'"),
    ("[x]", "'[x]'"), ("*a", "'*a'"), ("tab\there: x", '"tab\\there: x"'),
])
def test_scalar_styles(text, expected):
    assert isc.go_yaml_marshal({"k": text}) == f"k: {expected}\n".encode()


def test_empty_string_and_multiline():
    assert isc.go_yaml_marshal({"k": ""}) == b'k: ""\n'
    assert isc.go_yaml_marshal({"k": "a\nb\n"}) == b"k: |\n  a\n  b\n"
    assert isc.go_yaml_marshal({"k": "a\nb"}) == b"k: |-\n  a\n  b\n"


def test_long_options_fold_at_80_columns():
    opts = "--model meta-llama/Meta-Llama-3-8B --enable-sleep-mode --gpu-memory-utilization 0.4 --max-model-len 2048"
    out = isc.go_yaml_marshal({"options": opts}).decode()
    lines = out.splitlines()
    assert len(lines) == 2 and lines[1].startswith("  ")
    assert " ".join([lines[0][len("options: "):], lines[1].strip()]) == opts      # folding only replaces blanks
    assert len(lines[0]) > 80 and len(lines[0].rsplit(" ", 1)[0]) <= 80             # breaks at the first blank past col 80


def test_natural_key_order():
    assert isc.sorted_keys(["a10", "a9", "a1", "B", "_x", "a", "1", "10", "2"]) == \
        ["_x", "1", "2", "10", "B", "a", "a1", "a9", "a10"]   # "_" has no digit run: its number is 0 < 1


def test_instance_id_shape_and_sensitivity():
    cfg, iid = isc.config_inference_server("isc-a", 8005, "--model m --enable-sleep-mode",
                                           {"VLLM_SERVER_DEV_MODE": "1"}, {"team": "x"}, None, ["GPU-aa", "GPU-bb"])
    assert cfg == {"options": "--model m --enable-sleep-mode --port 8005", "gpu_uuids": ["GPU-aa", "GPU-bb"],
                   "env_vars": {"VLLM_SERVER_DEV_MODE": "1"},
                   "annotations": {"isc-name": "isc-a", "inference-port": "8005"}}
    assert iid[0] == "I" and iid[-1] == "i" and len(iid) == 45 and "=" not in iid
    body = b'env_vars:\n  VLLM_SERVER_DEV_MODE: "1"\nlabels:\n  team: x\noptions: --model m --enable-sleep-mode\nport: 8005\n'
    want = "I" + base64.urlsafe_b64encode(hashlib.sha256(body + b";gpus=GPU-aa,GPU-bb").digest()).rstrip(b"=").decode() + "i"
    assert iid == want
    # the ISC *name* is not hashed (two ISCs with equal model-server config share sleepers); GPUs, order included, are
    assert isc.config_inference_server("other", 8005, "--model m --enable-sleep-mode", {"VLLM_SERVER_DEV_MODE": "1"},
                                       {"team": "x"}, None, ["GPU-aa", "GPU-bb"])[1] == iid
    assert isc.config_inference_server("isc-a", 8005, "--model m --enable-sleep-mode", {"VLLM_SERVER_DEV_MODE": "1"},
                                       {"team": "x"}, None, ["GPU-bb", "GPU-aa"])[1] != iid
    assert isc.config_inference_server("isc-a", 8006, "--model m --enable-sleep-mode", {"VLLM_SERVER_DEV_MODE": "1"},
                                       {"team": "x"}, None, ["GPU-aa", "GPU-bb"])[1] != iid
    # no GPUs: ";gpus=" is still hashed and gpu_uuids is omitted from the body (omitempty)
    cfg0, _ = isc.config_inference_server("n", 1, "")
    assert "gpu_uuids" not in cfg0 and cfg0["options"] == " --port 1"
    with pytest.raises(ValueError):
        isc.config_inference_server("n", 0)


def test_instance_id_from_manifest_spec():
    spec = {"modelServerConfig": {"port": 8005, "options": "--model m"}, "launcherConfigName": "lc"}
    assert isc.instance_id(spec, ["G"]) == isc.config_inference_server("x", 8005, "--model m", gpu_uuids=["G"])[1]


def test_marshal_reproduces_the_references_generated_crds():
    """config/crd/*.yaml were written by controller-gen through sigs.k8s.io/yaml: parse them, marshal them again with the
    restatement, expect the same bytes — key order, folding at 80 columns, quoting of bool/number-like strings, literal
    blocks, indentless sequences.  The three files are stored xz-compressed under tests/golden/crd/."""
    import glob
    import lzma
    import os

    import yaml

    files = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "crd", "*.yaml.xz")))
    lines = 0
    for f in files:
        with lzma.open(f, "rt") as fh:
            text = fh.read()
        assert text.startswith("---\n")
        assert "---\n" + isc.go_yaml_marshal(yaml.safe_load(text)).decode() == text, os.path.basename(f)
        lines += text.count("\n")
    assert len(files) == 3 and lines > 8000


# ---- "same ID => wake" (selectBestLauncherPod, inference-server.go:680-785) over the launcher REST's JSON ----------------------
def _inst(iid, port, status="running"):
    return {"instance_id": iid, "status": status, "revision": 1, "options": f"--model m --port {port}", "annotations": {"isc-name": "x", "inference-port": str(port)}}


def _launcher(*insts):
    return {"revision": len(insts), "total_instances": len(insts), "running_instances": sum(1 for i in insts if i["status"] == "running"), "instances": list(insts)}


def test_select_launcher_priorities_and_port_conflicts():
    from fma_b200 import isc

    me, other = "Iminei", "Iotheri"
    # priority 1: the launcher that already holds MY instance wins over one that merely has room
    assert isc.select_launcher([("l-room", _launcher()), ("l-mine", _launcher(_inst(me, 8005), _inst(other, 8006)))], me, 8005, 1) == ("l-mine", True, False)
    # a stopped instance with my id is not a sleeper; the launcher still has room for one more (2 instances > max_others=1 -> no room)
    assert isc.select_launcher([("l", _launcher(_inst(me, 8005, "stopped")))], me, 8005, 1) == ("l", False, False)
    assert isc.select_launcher([("l", _launcher(_inst(me, 8005, "stopped"), _inst(other, 8006)))], me, 8005, 1) == (None, False, False)
    # another instance already listens on my port: skip that launcher
    assert isc.select_launcher([("l-conflict", _launcher(_inst(other, 8005))), ("l-free", _launcher())], me, 8005, 1) == ("l-free", False, False)
    # an instance without a usable port annotation poisons its launcher
    bad = _inst(other, 8006); bad["annotations"] = {"isc-name": "x"}
    assert isc.select_launcher([("l-bad", _launcher(bad))], me, 8005, 1) == (None, False, False)
    bad["annotations"]["inference-port"] = "80_05"
    assert isc.select_launcher([("l-bad", _launcher(bad))], me, 8005, 1) == (None, False, False)
    # not-ready launchers: retry instead of creating a new launcher, unless somebody else qualifies
    assert isc.select_launcher([("l-nr", None)], me, 8005, 1) == (None, False, True)
    assert isc.select_launcher([("l-nr", None), ("l-free", _launcher())], me, 8005, 1) == ("l-free", False, False)


def test_plan_actuation_from_isc_to_wake_or_create():
    from fma_b200 import isc

    spec = {"modelServerConfig": {"port": 8005, "options": "--model meta-llama/Llama-3-8B --enable-sleep-mode", "env_vars": {"VLLM_SERVER_DEV_MODE": "1"}},
            "launcherConfigName": "lc"}
    gpus = ["GPU-0a", "GPU-0b"]
    iid = isc.instance_id(spec, gpus)
    assert iid.startswith("I") and iid.endswith("i") and len(iid) == 45
    cfg, iid2 = isc.config_inference_server("my-isc", 8005, spec["modelServerConfig"]["options"], spec["modelServerConfig"]["env_vars"], gpu_uuids=gpus)
    assert iid2 == iid and cfg["annotations"] == {"isc-name": "my-isc", "inference-port": "8005"}
    # nothing there yet -> create on the launcher with room; the created instance (the launcher echoes id + annotations) then sleeps -> wake
    plan = isc.plan_actuation([("launcher-0", _launcher())], spec, gpus)
    assert plan == {"action": "create", "launcher": "launcher-0", "instance_id": iid, "port": 8005}
    mine = {"instance_id": iid, "status": "running", "revision": 1, **cfg}
    assert isc.plan_actuation([("launcher-0", _launcher(mine))], spec, gpus)["action"] == "wake"
    # different GPUs -> different ID -> my port is taken by "another" instance on that launcher -> elsewhere / new launcher
    assert isc.plan_actuation([("launcher-0", _launcher(mine))], spec, ["GPU-0c"]) == {"action": "new_launcher", "launcher": None, "instance_id": isc.instance_id(spec, ["GPU-0c"]), "port": 8005}
    assert isc.plan_actuation([("launcher-0", None)], spec, gpus)["action"] == "retry"
