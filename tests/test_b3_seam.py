"""not-gpu: B200Supervisor behind the REAL reference server, replayed from recorded exchanges.

tests/golden/b3_seam.json holds what the unmodified reference server did with the 3-line supervisor_factory hook of
INTEGRATION.md applied (oracle/make_b3_golden.py records it through tests/b3_driver.py): for every call, the request
body the reference's client codec produced and the status code and JSON body the reference server answered.  This
pins seam B3 (SURVEY.md §8(b)): construction from KT_DISTRIBUTED_CONFIG alone, callable from the KT_* environment,
raw `{"data": b64}` bodies in, per-rank `{"data": b64}` out, `workers=` errors, allow-list errors.  Each recorded
request goes into B200Supervisor.call the way the server calls it, exceptions are packaged by the oracle's
restatement of the server's handler, and the answer must equal the recorded one.  The device layer is a torch-CPU
stub here; tests/test_gpu_api.py::test_b3_* run the same contract against the real kernels."""
import json
import os

import pytest
import torch

from conftest import REPO
from oracle import ref_dispatch

GOLDEN = os.path.join(REPO, "tests", "golden", "b3_seam.json")


def _t(dtype, shape, seed=0):
    return {"tensor": {"dtype": dtype, "shape": shape, "seed": seed}}


# the deployments the recorded exchanges come from: callable, distributed config, allow-list, calls
RUNS = {
    "double_x4": {"callable": "double", "distributed_config": {"distribution_type": "b200", "num_proc": 4, "self_check": False},
                  "calls": [{"args": [_t("float32", [1003])]}, {"args": [_t("float32", [3])]},
                            {"args": [_t("float32", [10, 7], 3)]},
                            {"args": [_t("float32", [1003])], "kwargs": {"workers": [10]}},
                            {"args": [_t("float32", [1003])], "kwargs": {"workers": [1.5]}},
                            {"args": [_t("float32", [1003])], "kwargs": {"workers": "any"}}]},
    "double_2x2": {"callable": "double",
                   "distributed_config": {"distribution_type": "b200", "num_proc": 2, "quorum_workers": 2, "self_check": False},
                   "calls": [{"args": [_t("float32", [1003])]}, {"args": [_t("float32", [1003])], "kwargs": {"workers": [1]}},
                             {"args": [_t("float32", [1003])], "kwargs": {"workers": [7]}}]},
    "double_json_only": {"callable": "double", "allowed": "json",
                         "distributed_config": {"distribution_type": "b200", "num_proc": 2, "self_check": False},
                         "calls": [{"args": [_t("float32", [8])], "serialization": "pickle"}]},
    "scaler_x3": {"callable": "Scaler", "init_args": {"tag": "t"},
                  "distributed_config": {"distribution_type": "b200", "num_proc": 3, "self_check": False},
                  "calls": [{"method": "triple", "args": [_t("int64", [130])]}, {"method": "nope", "args": []}]},
    "affine_x2": {"callable": "affine", "distributed_config": {"distribution_type": "b200", "num_proc": 2, "self_check": False},
                  "calls": [{"args": [_t("float32", [1001], 5), 0.1], "kwargs": {"beta": 0.3}},
                            {"args": [_t("int64", [130]), 0.5, 1]}]},
}


def _recorded(name):
    with open(GOLDEN) as f:
        run = json.load(f)["runs"][name]
    assert run["config"] == json.loads(json.dumps(RUNS[name])), \
        f"{name}: RUNS changed since the recording; regenerate with oracle/make_b3_golden.py"
    return run


def _same(got, want):
    if isinstance(want, torch.Tensor):
        return isinstance(got, torch.Tensor) and got.dtype == want.dtype and got.shape == want.shape and \
            torch.equal(got.reshape(-1).view(torch.uint8), want.reshape(-1).view(torch.uint8))
    if isinstance(want, list):
        return isinstance(got, list) and len(got) == len(want) and all(_same(g, w) for g, w in zip(got, want))
    return got == want


def _run(name, monkeypatch):
    """Deploy RUNS[name] the way the reference server does, replay its recorded requests, check every answer
    against the recorded one, and return what a client decodes from the answers."""
    import b3_driver
    from kubetorch_b200.serving.b200_supervisor import B200Supervisor
    from kubetorch_b200.serving.supervisors import Request

    run = _recorded(name)
    cfg = RUNS[name]
    for k, v in {"POD_NAMESPACE": "kubetorch", "POD_NAME": "b3-pod", "POD_IP": "localhost", "LOCAL_IPS": "localhost",
                 "KT_SERVICE_NAME": "b3", "KT_FILE_PATH": os.path.join(REPO, "tests"), "KT_MODULE_NAME": "b3_user_module",
                 "KT_CLS_OR_FN_NAME": cfg["callable"], "KT_INIT_ARGS": json.dumps(cfg.get("init_args")),
                 "KT_ALLOWED_SERIALIZATION": cfg.get("allowed", "json,pickle"),
                 "KT_DISTRIBUTED_CONFIG": json.dumps(cfg["distributed_config"])}.items():
        monkeypatch.setenv(k, v)
    stub = b3_driver.stub_device()
    monkeypatch.setattr(B200Supervisor, "_load_device", lambda self: stub)
    kwargs = json.loads(os.environ["KT_DISTRIBUTED_CONFIG"])
    kwargs.pop("distribution_type")                    # supervisor_factory(distribution_type, **rest)
    sup = B200Supervisor(**kwargs)
    sup.setup()
    records = []
    try:
        for ex in run["exchanges"]:
            fn_name, _, method = ex["path"].strip("/").partition("/")
            try:
                answer = sup.call(Request({"X-Serialization": ex["serialization"], "X-Request-ID": "b3"}), fn_name,
                                  method or None, json.loads(json.dumps(ex["request"])))
                status, answer = 200, json.loads(json.dumps(answer))      # the server's JSON response body
            except Exception as e:  # noqa: BLE001 - the server's generic exception handler
                status, answer = ref_dispatch.package_exception(e)
            assert status == ex["status_code"], (name, ex["path"], status, answer)
            rec = {"status_code": status}
            if status == 200:
                res = ref_dispatch.deserialize_response(answer, ex["serialization"])
                assert _same(res, ref_dispatch.deserialize_response(ex["response"], ex["serialization"])), (name, ex["path"])
                rec["result"] = [{"dtype": str(t.dtype), "shape": list(t.shape), "data": t.reshape(-1).tolist()}
                                 if isinstance(t, torch.Tensor) else t for t in res] if isinstance(res, list) else res
            else:
                for k, v in ex["response"].items():
                    assert answer.get(k) == v, (name, ex["path"], k, answer.get(k), v)
                rec["error"] = {k: answer.get(k) for k in ("error_type", "message", "pod_name", "detail") if k in answer}
            records.append(rec)
    finally:
        sup.cleanup()
    assert [list(c) for c in stub.calls] == run["device_calls"], name
    return {"records": records, "device_calls": stub.calls}


def _make(spec):
    g = torch.Generator().manual_seed(spec["tensor"].get("seed", 0))
    dt = getattr(torch, spec["tensor"]["dtype"])
    if dt.is_floating_point:
        return torch.randn(spec["tensor"]["shape"], generator=g).to(dt)
    return torch.randint(-1000, 1000, spec["tensor"]["shape"], generator=g, dtype=dt)


def _shards(x, world):
    ch = x.chunk(world)
    return [ch[r] if r < len(ch) else x[:0] for r in range(world)]


def test_reference_server_drives_b200_supervisor_with_raw_pickle_bodies(monkeypatch):
    x, small = _t("float32", [1003]), _t("float32", [3])
    out = _run("double_x4", monkeypatch)
    recs = out["records"]
    for rec, spec in zip(recs[:3], (x, small, _t("float32", [10, 7], 3))):
        assert rec["status_code"] == 200, rec
        want = [s * 2 for s in _shards(_make(spec), 4)]
        assert len(rec["result"]) == 4
        for got, w in zip(rec["result"], want):
            assert got["dtype"] == str(w.dtype) and got["shape"] == list(w.shape)
            assert got["data"] == w.reshape(-1).tolist()
    # the reference's selector errors, through the reference's own exception handler (recorded: workers_bad_index/spec)
    assert recs[3]["status_code"] == 400 and recs[3]["error"]["error_type"] == "ValueError"
    assert recs[3]["error"]["message"] == "Worker index 10 out of range. Valid range: 0-0"
    assert recs[4]["status_code"] == 400 and recs[4]["error"]["message"] == (
        "Invalid worker specification: 1.5. Must be an IP address, integer index, or numeric string.")
    assert recs[5]["status_code"] == 200 and len(recs[5]["result"]) == 4      # "any" = the coordinator's local ranks
    assert ("map_host_multi", 4) in [tuple(c) for c in out["device_calls"]]


def test_reference_server_multi_node_config_and_workers_subset(monkeypatch):
    """quorum_workers=2 x num_proc=2 (the recorded mp_double_* shape): `workers=[1]` returns node 1's ranks only,
    which keep their GLOBAL rank / world size (recorded shapes [(251,), (250,)])."""
    x = _t("float32", [1003])
    out = _run("double_2x2", monkeypatch)
    full, sub, bad = out["records"]
    want = [s * 2 for s in _shards(_make(x), 4)]
    assert [r["shape"] for r in full["result"]] == [[251], [251], [251], [250]]
    assert [r["shape"] for r in sub["result"]] == [[251], [250]]
    assert sub["result"][0]["data"] == want[2].tolist() and sub["result"][1]["data"] == want[3].tolist()
    assert bad["status_code"] == 400 and bad["error"]["message"] == "Worker index 7 out of range. Valid range: 0-1"


def test_reference_server_allow_list_json_mode_and_class_callable(monkeypatch):
    out = _run("double_json_only", monkeypatch)
    rec = out["records"][0]
    assert rec["status_code"] == 400
    assert "Serialization format 'pickle' not allowed. Allowed formats: ['json']" in json.dumps(rec["error"])
    # a class: instance built from KT_INIT_ARGS, method from the URL, kwargs-bound parameters of an affine op
    out = _run("scaler_x3", monkeypatch)
    ok, missing = out["records"]
    want = [s * 3 for s in _shards(_make(_t("int64", [130])), 3)]
    assert [r["data"] for r in ok["result"]] == [w.tolist() for w in want]
    assert missing["status_code"] == 404 and "Method 'nope' not found in class 'Scaler'" in json.dumps(missing["error"])
    out = _run("affine_x2", monkeypatch)
    rec, bad = out["records"]
    want = [s * 0.1 + 0.3 for s in _shards(_make(_t("float32", [1001], 5)), 2)]
    assert [r["data"] for r in rec["result"]] == [w.tolist() for w in want]
    assert bad["status_code"] == 422 and bad["error"]["error_type"] == "TypeError"   # non-integral alpha on an int tensor
