"""SURVEY §8 row f1: the sdwui-compatible REST worker (server/sdapi.py), driven over real HTTP by
 (1) this repo's `Worker` (which keeps the reference's HTTP transport for remote nodes), and
 (2) the UNMODIFIED reference `Worker`: the requests it sent and what it made of the replies are stored golden data
     (tests/golden/gen_rest_worker_golden.py -> tests/golden/rest_worker_golden.json), replayed here over HTTP.
The executor is replaced by a deterministic double: this file tests the wire contract, not the arithmetic."""
import base64
import hashlib
import io
import json
import os
import socket
import threading
import time
import types

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REST_GOLDEN = os.path.join(HERE, "golden", "rest_worker_golden.json")


class EngineDouble:
    """same call surface as b200sd.SDEngine, images are a pure function of (seed, tokens, size)"""

    def __init__(self):
        self.interrupted = False
        self.clip_cfg = types.SimpleNamespace(vocab=1000)
        self.calls = []

    @staticmethod
    def _images(seed, tok, b, h, w, extra=0):
        out = []
        for i in range(b):
            g = torch.Generator().manual_seed(int(seed) + i + 1000 * int(tok[i % tok.shape[0]].sum()) + extra)
            out.append(torch.randint(0, 256, (h, w, 3), generator=g, dtype=torch.uint8))
        return torch.stack(out)

    def txt2img(self, tok, neg, seed, steps, cfg_scale, height, width, sampler, scheduler=None):
        self.calls.append(("txt2img", int(seed), int(tok.shape[0]), steps, sampler))
        return self._images(seed, tok, tok.shape[0], height, width)

    def img2img(self, tok, neg, seed, init_u8, denoising_strength, steps, cfg_scale, sampler="DDIM", scheduler=None, latmask=None, inpainting_fill=1):
        self.calls.append(("img2img", int(seed), int(tok.shape[0]), steps, float(denoising_strength)))
        b, h, w, _ = init_u8.shape
        return self._images(seed, tok, b, h, w, extra=int(init_u8.sum()) % 997)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


@pytest.fixture(scope="module")
def server():
    import uvicorn
    from server.sdapi import create_app
    eng = EngineDouble()
    port = _free_port()
    app = create_app(lambda device: eng, [0])
    cfg = uvicorn.Config(app, host="127.0.0.1", port=port, log_level="error")
    srv = uvicorn.Server(cfg)
    t = threading.Thread(target=srv.run, daemon=True)
    t.start()
    for _ in range(200):
        if srv.started:
            break
        time.sleep(0.05)
    assert srv.started
    yield port, eng
    srv.should_exit = True
    t.join(timeout=5)


def _decode(b64png):
    from PIL import Image
    return np.asarray(Image.open(io.BytesIO(base64.b64decode(b64png))))


def reply_digest(path, body):
    """what the REST golden file keeps of a reply: images as the SHA-1 of their decoded pixels, and of /memory (live
    numbers, and 'cuda' depends on the machine) only whether the fields the reference Worker reads are there"""
    if path.endswith("/memory"):
        cuda = body.get("cuda", {})
        return {"keys": sorted(body), "cuda_readable": "error" in cuda or {"free", "total"} <= set(cuda.get("system", {}))}
    if isinstance(body, dict) and "images" in body:
        return dict(body, images=[hashlib.sha1(_decode(s).tobytes()).hexdigest() for s in body["images"]])
    return body


PAYLOAD = {"prompt": "a probe", "negative_prompt": "", "seed": 31, "subseed": 7, "subseed_strength": 0, "batch_size": 2,
           "n_iter": 1, "steps": 4, "width": 64, "height": 64, "sampler_name": "DDIM", "cfg_scale": 7.0,
           "s_tmax": float("inf"), "alwayson_scripts": {}}


def _expected(eng, payload, extra=0):
    from b200sd.factory import synthetic_tokens
    tok = synthetic_tokens([payload["prompt"]] * payload["batch_size"], eng.clip_cfg.vocab)
    return eng._images(payload["seed"], tok, payload["batch_size"], payload["height"], payload["width"], extra)


def test_our_worker_drives_the_rest_server(server):
    port, eng = server
    from scripts.spartan import pmodels, shared
    from scripts.spartan.worker import State, Worker
    shared.benchmark_payload = pmodels.Benchmark_Payload()  # what World.load_config() installs
    w = Worker(address="127.0.0.1", port=port, label="b200box", verify_remotes=False, avg_ipm=600.0)
    assert w.reachable()
    w.benchmarked = True
    w.request(dict(PAYLOAD), {"sd_model_checkpoint": "m.safetensors", "sd_vae": None}, True)
    r = w.response
    assert w.state == State.IDLE and w.jobs_requested == 1 and w.loaded_model == "m.safetensors"
    assert set(r) == {"images", "parameters", "info"} and len(r["images"]) == 2
    info = json.loads(r["info"])
    assert info["all_seeds"] == [31, 32] and info["all_subseeds"] == [7, 8] and len(info["infotexts"]) == 2
    want = _expected(eng, PAYLOAD)
    for i in range(2):
        assert np.array_equal(_decode(r["images"][i]), want[i].numpy())
    assert eng.calls[-1] == ("txt2img", 31, 2, 4, "DDIM")
    assert w.available_models() == ["b200sd-synthetic.safetensors [00000000]"] or len(w.available_models()) == 1


def test_raw_routes_and_img2img(server):
    port, eng = server
    import requests
    base = f"http://127.0.0.1:{port}/sdapi/v1"
    mem = requests.get(f"{base}/memory", timeout=5).json()
    assert "cuda" in mem and "ram" in mem  # no GPU here: cuda carries an 'error' field, as sdwui does
    assert requests.get(f"{base}/script-info", timeout=5).json() == []
    assert requests.post(f"{base}/options", json={"sd_model_checkpoint": "x", "sd_vae": "y"}, timeout=5).status_code == 200
    assert requests.get(f"{base}/options", timeout=5).json() == {"sd_model_checkpoint": "x", "sd_vae": "y"}
    for route in ("interrupt", "refresh-checkpoints", "refresh-loras", "server-restart"):
        assert requests.post(f"{base}/{route}", timeout=5).status_code == 200
    models = requests.get(f"{base}/sd-models", timeout=5).json()
    assert isinstance(models, list) and "title" in models[0]
    # img2img: the API's wire format for init images is base64 PNG (reference worker.py:365-373)
    from PIL import Image
    g = torch.Generator().manual_seed(5)
    init = torch.randint(0, 256, (64, 64, 3), generator=g, dtype=torch.uint8)
    buf = io.BytesIO()
    Image.fromarray(init.numpy()).save(buf, format="PNG")
    payload = dict(PAYLOAD, s_tmax=None, init_images=["data:image/png;base64," + base64.b64encode(buf.getvalue()).decode()],
                   denoising_strength=0.6, batch_size=1)
    r = requests.post(f"{base}/img2img", json=payload, timeout=30)
    assert r.status_code == 200
    assert eng.calls[-1][0] == "img2img" and eng.calls[-1][4] == pytest.approx(0.6)
    want = _expected(eng, payload, extra=int(init.sum()) % 997)
    assert np.array_equal(_decode(r.json()["images"][0]), want[0].numpy())
    assert requests.post(f"{base}/img2img", json=dict(PAYLOAD, s_tmax=None), timeout=5).status_code == 404  # no init image


def test_api_auth():
    from fastapi.testclient import TestClient
    from server.sdapi import create_app
    c = TestClient(create_app(lambda device: EngineDouble(), [0], api_auth="user:secret"))
    assert c.get("/sdapi/v1/memory").status_code == 401
    assert c.get("/sdapi/v1/memory", auth=("user", "wrong")).status_code == 401
    assert c.get("/sdapi/v1/memory", auth=("user", "secret")).status_code == 200


def test_requests_are_bounded_and_restart_waits_for_the_running_generation():
    """ADVICE r1: a client must not be able to walk the device out of memory by varying sizes (every distinct batch / size
    builds buffers and graphs), and /server-restart must not pull the engine from under a generation in flight"""
    from fastapi.testclient import TestClient
    from server import sdapi
    from server.sdapi import create_app

    class Slow(EngineDouble):
        def __init__(self):
            super().__init__()
            self.running = threading.Event()
            self.release = threading.Event()

        def txt2img(self, *a, **k):
            self.running.set()
            assert self.release.wait(10)
            return super().txt2img(*a, **k)

    eng = Slow()
    built = []

    def factory(device):
        built.append(device)
        return eng
    app = create_app(factory, [0])
    c = TestClient(app)
    ok = dict(PAYLOAD, s_tmax=None)
    for bad in ({"batch_size": 0}, {"batch_size": sdapi.MAX_BATCH + 1}, {"n_iter": 0}, {"steps": 0}, {"steps": 151},
                {"width": sdapi.MAX_SIDE + 64}, {"height": 32}, {"width": 100}, {"batch_size": "many"}):
        assert c.post("/sdapi/v1/txt2img", json=dict(ok, **bad)).status_code == 422, bad
    assert eng.calls == [] and built == []     # nothing reached the executor, no engine was even built
    # a generation in flight holds its device's lock: the restart waits for it, then drops the engine
    import scripts.spartan.local_worker as lw
    evicted = []
    orig = lw.LocalGPUWorker.restart
    lw.LocalGPUWorker.restart = lambda self: evicted.append(eng.release.is_set()) or True
    try:
        res = {}
        t = threading.Thread(target=lambda: res.setdefault("gen", c.post("/sdapi/v1/txt2img", json=ok)))
        t.start()
        assert eng.running.wait(10)
        r = threading.Thread(target=lambda: res.setdefault("restart", c.post("/sdapi/v1/server-restart")))
        r.start()
        time.sleep(0.3)
        assert evicted == []            # still waiting for the generation
        eng.release.set()
        t.join(10)
        r.join(10)
    finally:
        lw.LocalGPUWorker.restart = orig
    assert res["gen"].status_code == 200 and res["restart"].status_code == 200
    assert evicted == [True]            # the restart ran after the generation had been released


def test_unmodified_reference_worker_drives_the_rest_server(server):
    """the requests the reference Worker sent, replayed: the server answers each as it did when the reference drove it,
    so the reference would reach the same state and images it did then"""
    port, eng = server
    import requests
    with open(REST_GOLDEN) as f:
        golden = json.load(f)
    assert [e["path"].rsplit("/", 1)[1] for e in golden["exchange"]] == ["memory", "memory", "options", "txt2img", "sd-models"]
    for e in golden["exchange"]:
        r = requests.request(e["method"], f"http://127.0.0.1:{port}{e['path']}", json=e["json"], timeout=30)
        assert r.status_code == e["status"], e["path"]
        assert reply_digest(e["path"], r.json()) == e["reply"], e["path"]
    assert eng.calls[-1] == ("txt2img", 31, 2, 4, "DDIM")
    out = golden["reference_worker"]
    assert out["reachable"] and out["state"] == "IDLE" and out["n_images"] == 2
    assert out["all_seeds"] == [31, 32] and out["all_subseeds"] == [7, 8]
    want = _expected(eng, PAYLOAD)
    assert out["image_sha1"] == [hashlib.sha1(want[i].numpy().tobytes()).hexdigest() for i in range(2)]
    assert out["loaded_model"] == "m.safetensors" and len(out["models"]) == 1
