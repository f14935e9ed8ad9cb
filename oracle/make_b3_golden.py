"""Generate tests/golden/b3_seam.json: the UNMODIFIED reference server driving B200Supervisor.

TEST INFRASTRUCTURE.  Needs the reference tree (oracle/make_golden.py:REFERENCE).  For every configuration in
tests/test_b3_seam.py:RUNS it runs tests/b3_driver.py — the reference's FastAPI app under TestClient with the
supervisor_factory hook of INTEGRATION.md, device layer stubbed with torch CPU ops — and stores each exchange: the
request body the reference client produced, and the status code and JSON body the reference server answered
(tracebacks dropped).  tests/test_b3_seam.py replays the requests into B200Supervisor and compares.

Usage:  python oracle/make_b3_golden.py            # regenerates tests/golden/b3_seam.json
"""
from __future__ import annotations

import json
import os
import subprocess
import sys
import tempfile

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [REPO, os.path.join(REPO, "tests")]

from oracle.make_golden import REFERENCE, STUB  # noqa: E402
from test_b3_seam import GOLDEN, RUNS  # noqa: E402


def record(cfg: dict) -> dict:
    work = tempfile.mkdtemp(prefix="kt_b3_")
    with open(os.path.join(work, "websocket.py"), "w") as f:   # the one absent import of the reference (never used here)
        f.write(STUB)
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([work, REFERENCE, REPO])
    env["HOME"] = work
    env["PYTHONDONTWRITEBYTECODE"] = "1"
    p = subprocess.run([sys.executable, os.path.join(REPO, "tests", "b3_driver.py"), "--stub",
                        json.dumps(dict(cfg, repo=REPO))], env=env, cwd=work, capture_output=True, text=True, timeout=600)
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("B3RESULT ")]
    if p.returncode != 0 or not lines:
        raise SystemExit(p.stdout[-2000:] + p.stderr[-4000:])
    return dict(json.loads(lines[-1][len("B3RESULT "):]), config=cfg)


def main():
    if not os.path.isdir(REFERENCE):
        raise SystemExit(f"{REFERENCE} not found: the B3 goldens can only be regenerated where the reference is")
    runs = {}
    for name, cfg in RUNS.items():
        print(f"[make_b3_golden] {name} ...", flush=True)
        runs[name] = record(cfg)
    out = {"provenance": {"generator": "oracle/make_b3_golden.py",
                          "reference": "run-house/kubetorch @ 96fac95 (python_client v0.5.0), unmodified http_server "
                                       "under fastapi TestClient, supervisor_factory hook of INTEGRATION.md"},
           "runs": runs}
    with open(GOLDEN, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print(f"[make_b3_golden] wrote {GOLDEN}: {len(runs)} runs, {os.path.getsize(GOLDEN)} bytes")


if __name__ == "__main__":
    main()
