"""Child process of oracle/make_b3_golden.py, which records tests/golden/b3_seam.json (needs the reference tree).

Runs the UNMODIFIED reference server (kubetorch.serving.http_server:app under fastapi's TestClient, as the
reference's own tests/test_http_server.py:86-96 does) with ONE change: the 3-line hook INTEGRATION.md gives for
kubetorch/serving/supervisor_factory.py, applied by monkeypatching.  The server then builds B200Supervisor exactly
as it builds its own supervisors — `supervisor_factory(**json.loads(KT_DISTRIBUTED_CONFIG))`, callable from the
KT_* environment, RAW request bodies into SUPERVISOR.call — and the reference's CLIENT codecs
(_serialize_body / _deserialize_response) sit on both ends.  Prints every exchange: the request body the reference
client sent and the status and JSON body the reference server answered.  The device layer is stubbed with torch
CPU ops (`--stub`, what tests/test_b3_seam.py replays against); pass `--device` to run the real kernels."""
import json
import os
import sys


def stub_device():
    import torch

    from kubetorch_b200.device import ops as real

    class Stub:
        shard_bounds = staticmethod(real.shard_bounds)
        row_elems = staticmethod(real.row_elems)
        calls = []

        @staticmethod
        def device_count():
            return 8

        @staticmethod
        def ensure_init(devs):
            pass

        @staticmethod
        def synchronize(dev):
            pass

        @staticmethod
        def join_devices(root, devs):
            pass

        @staticmethod
        def is_pinned(t):
            return True

        @staticmethod
        def pinned_empty(shape, dtype, devices=None):
            return torch.empty(shape, dtype=dtype)

        @staticmethod
        def _apply(x, op, alpha, beta):
            if op == "identity":
                return x.clone()
            return x * alpha if op == "scale" else x * alpha + beta

        @classmethod
        def map_host_multi(cls, x, op, alpha=1.0, beta=0.0, out_host=None, devices=(0,), chunk_bytes=None):
            cls.calls.append(("map_host_multi", len(devices)))
            out_host.copy_(cls._apply(x, op, alpha, beta))
            return out_host

        @classmethod
        def map_host(cls, x, op, alpha=1.0, beta=0.0, out_host=None, device=0, chunk_bytes=None):
            cls.calls.append(("map_host", device))
            out_host.copy_(cls._apply(x, op, alpha, beta))
            return out_host

    return Stub


def main():
    mode = sys.argv[1]
    cfg = json.loads(sys.argv[2])
    os.environ["KT_LOG_STREAMING_ENABLED"] = "false"
    os.environ["KT_METRICS_ENABLED"] = "false"
    os.environ.update({
        "POD_NAMESPACE": "kubetorch", "POD_NAME": "b3-pod", "POD_IP": "localhost", "LOCAL_IPS": "localhost",
        "KT_SERVICE_NAME": "b3", "KT_FILE_PATH": os.path.join(cfg["repo"], "tests"), "KT_MODULE_NAME": "b3_user_module",
        "KT_CLS_OR_FN_NAME": cfg["callable"], "KT_INIT_ARGS": json.dumps(cfg.get("init_args")),
        "KT_ALLOWED_SERIALIZATION": cfg.get("allowed", "json,pickle"),
        "KT_DISTRIBUTED_CONFIG": json.dumps(cfg["distributed_config"]),
    })
    import torch
    from fastapi.testclient import TestClient

    import kubetorch.serving.supervisor_factory as ref_factory          # the REAL reference module
    from kubetorch.resources.callables.utils import build_call_body
    from kubetorch.serving.utils import _deserialize_response, _serialize_body

    original = ref_factory.supervisor_factory

    def supervisor_factory(distribution_type, *args, **kwargs):         # the hook of INTEGRATION.md §1
        if distribution_type == "b200":
            from kubetorch_b200.serving.b200_supervisor import B200Supervisor

            return B200Supervisor(*args, **kwargs)
        return original(distribution_type, *args, **kwargs)

    ref_factory.supervisor_factory = supervisor_factory
    stub = None
    if mode == "--stub":
        from kubetorch_b200.serving.b200_supervisor import B200Supervisor

        stub = stub_device()
        B200Supervisor._load_device = lambda self: stub

    from kubetorch.serving.http_server import app

    def tens(spec):
        g = torch.Generator().manual_seed(spec.get("seed", 0))
        dt = getattr(torch, spec["dtype"])
        if dt.is_floating_point:
            return torch.randn(spec["shape"], generator=g).to(dt)
        return torch.randint(-1000, 1000, spec["shape"], generator=g, dtype=dt)

    def resolve(v):
        if isinstance(v, dict) and "tensor" in v:
            return tens(v["tensor"])
        if isinstance(v, list):
            return [resolve(a) for a in v]
        return v

    out = []
    with TestClient(app, raise_server_exceptions=False) as client:
        for call in cfg["calls"]:
            args = resolve(call.get("args", []))
            ser = call.get("serialization", "pickle")
            body = _serialize_body(build_call_body(*args, **dict(call.get("kwargs") or {})), ser)
            url = f"/{cfg['callable']}" + (f"/{call['method']}" if call.get("method") else "")
            request = json.loads(json.dumps(body))        # what goes on the wire (the server may consume `body`)
            resp = client.post(url, json=body, headers={"X-Serialization": ser, "X-Request-ID": "b3"})
            response = resp.json()
            if resp.status_code != 200:
                response.pop("traceback", None)           # host-specific file paths, not part of the contract
            else:
                _deserialize_response(resp, ser)          # the reference client accepts the body
            out.append({"path": url, "serialization": ser, "request": request, "status_code": resp.status_code,
                        "response": response})
    print("B3RESULT " + json.dumps({"exchanges": out, "device_calls": stub.calls if stub else None}))


if __name__ == "__main__":      # the reference spawns workers for ITS supervisors; harmless here, kept for parity
    main()
