"""Drives a running sdwui-API worker server with the UNMODIFIED reference `Worker` class, in its own process because the
reference's module names (`scripts.spartan.*`) are the same as this repo's.

    python tests/ref_rest_probe.py <port> <reference checkout>       -> one JSON line on stdout

Used by tests/golden/gen_rest_worker_golden.py.
"""
import base64
import io
import json
import logging.handlers
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
REF = sys.argv[2]
tmp = tempfile.mkdtemp(prefix="refprobe_")
os.environ["HOSTSTUB_CONFIG_DIR"] = tmp
sys.path[:0] = [os.path.join(HERE, "hoststub"), REF]

import pydantic.v1  # noqa: E402

sys.modules["pydantic"] = pydantic.v1
_Orig = logging.handlers.RotatingFileHandler


class _Redirected(_Orig):
    def __init__(self, filename, *a, **k):
        super().__init__(os.path.join(tmp, os.path.basename(str(filename))), *a, **k)


logging.handlers.RotatingFileHandler = _Redirected

from scripts.spartan import pmodels, shared, worker  # noqa: E402  (the reference's)

logging.getLogger("distributed").setLevel(logging.CRITICAL + 1)
shared.benchmark_payload = pmodels.Benchmark_Payload()  # what World.load_config() installs (world.py:672-676)


def main():
    port = int(sys.argv[1])
    w = worker.Worker(address="127.0.0.1", port=port, label="b200box", verify_remotes=False, avg_ipm=600.0)
    out = {"reference_file": worker.__file__, "reachable": bool(w.reachable())}
    w.benchmarked = True
    payload = {"prompt": "a probe", "negative_prompt": "", "seed": 31, "subseed": 7, "subseed_strength": 0, "batch_size": 2,
               "n_iter": 1, "steps": 4, "width": 64, "height": 64, "sampler_name": "DDIM", "cfg_scale": 7.0,
               "s_tmax": float("inf"), "alwayson_scripts": {}}
    w.request(dict(payload), {"sd_model_checkpoint": "m.safetensors", "sd_vae": None}, True)
    r = w.response
    out["state"] = w.state.name
    out["n_images"] = len(r["images"])
    info = json.loads(r["info"])
    out["all_seeds"] = info["all_seeds"]
    out["all_subseeds"] = info["all_subseeds"]
    from PIL import Image
    import hashlib
    import numpy as np
    out["image_sha1"] = [hashlib.sha1(np.asarray(Image.open(io.BytesIO(base64.b64decode(s)))).tobytes()).hexdigest()
                         for s in r["images"]]
    out["loaded_model"] = w.loaded_model
    out["models"] = w.available_models()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
