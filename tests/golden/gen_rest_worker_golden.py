"""Generates tests/golden/rest_worker_golden.json: the UNMODIFIED reference `Worker` (scripts/spartan/worker.py of a
papuSpartan/stable-diffusion-webui-distributed checkout) drives this repo's sdwui-API worker server (server/sdapi.py,
executor = the deterministic EngineDouble of tests/test_rest_worker_cpu.py) over real HTTP.  Every request it sends
is recorded with the server's reply, together with what the reference Worker made of those replies.

    python tests/golden/gen_rest_worker_golden.py <reference checkout>

tests/test_rest_worker_cpu.py replays the recorded requests and checks that the server still answers them the same.
"""
import json
import os
import subprocess
import sys
import threading
import time

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
sys.path[:0] = [TESTS, os.path.join(TESTS, "hoststub"), os.path.join(ROOT, "stable-diffusion-webui-distributed_b200")]

import uvicorn  # noqa: E402
from starlette.responses import Response  # noqa: E402

from server.sdapi import create_app  # noqa: E402
from test_rest_worker_cpu import EngineDouble, _free_port, reply_digest  # noqa: E402


def main():
    ref = os.path.abspath(sys.argv[1])
    app = create_app(lambda device: EngineDouble(), [0])
    exchange = []

    @app.middleware("http")
    async def record(request, call_next):
        body = await request.body()
        response = await call_next(request)
        data = b"".join([chunk async for chunk in response.body_iterator])
        path = request.url.path
        exchange.append({"method": request.method, "path": path, "json": json.loads(body) if body else None,
                         "status": response.status_code, "reply": reply_digest(path, json.loads(data))})
        return Response(content=data, status_code=response.status_code, headers=dict(response.headers))

    port = _free_port()
    srv = uvicorn.Server(uvicorn.Config(app, host="127.0.0.1", port=port, log_level="error"))
    t = threading.Thread(target=srv.run, daemon=True)
    t.start()
    while not srv.started:
        time.sleep(0.05)
    p = subprocess.run([sys.executable, os.path.join(TESTS, "ref_rest_probe.py"), str(port), ref], capture_output=True,
                       text=True, timeout=120)
    srv.should_exit = True
    t.join(timeout=5)
    if p.returncode != 0:
        raise SystemExit(p.stderr[-2000:])
    worker = json.loads(p.stdout.strip().splitlines()[-1])
    assert worker.pop("reference_file").startswith(ref), "the probe imported a Worker from outside the reference"
    golden = {"_meta": {"reference": "papuSpartan/stable-diffusion-webui-distributed @ 8fd65ebd",
                        "generator": "tests/golden/gen_rest_worker_golden.py"},
              "reference_worker": worker, "exchange": exchange}
    out = os.path.join(HERE, "rest_worker_golden.json")
    with open(out, "w") as f:
        json.dump(golden, f, indent=1, sort_keys=True)
    print("wrote", out, [(e["method"], e["path"], e["status"]) for e in exchange])


if __name__ == "__main__":
    main()
