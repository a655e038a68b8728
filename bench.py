#!/usr/bin/env python
"""bench.py — images/sec of the batch-sharded SD1.5 txt2img path (BASELINE.json metric) on N GPUs of one node.

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # BASELINE config 1 on the box's host cores: HTTP-dispatched CPU workers
    python bench.py --workload img2img        # BASELINE config 3
    python bench.py --sweep 1,2,4,8,16,32,64  # BASELINE config 5 (per-GPU batch sweep), one JSON line with a list
    python bench.py --dump-outputs DIR        # also write the last timed step's images to DIR as .npy, to compare builds

One "step" = one whole txt2img request of the per-GPU batch: CLIP encode, 20 DDIM timesteps (19 UNet evaluations
on [cond | uncond]) and the VAE decode to uint8, plus — for N > 1 — the single NCCL all-gather of the images.
Ranks own disjoint image indices (seed + k), weights are replicated, there is no per-step collective: scaling "weak"
(per-GPU batch fixed at --per-gpu-batch, default 32 = BASELINE.json configs[1]'s batch on one GPU).

  value          images/s with prompts/noise already resident in HBM (device-timed with CUDA events, max over ranks)
  e2e            the same request issued through the reference-facing plugin surface — DistributedScript hooks driving a
                 LocalGPUWorker.request() — from HOST buffers: prompt strings/tokens and per-image CPU-RNG noise are
                 uploaded, decoded uint8 images are copied back into `worker.response` inside the timed region
  world_e2e      rank 0 alone drives ONE DistributedScript whose World holds a LocalGPUWorker for EVERY GPU of the job
                 (the north-star design: one request's batch sharded by World.optimize_jobs, one thread per job,
                 reference scripts/distributed.py:288-318, collector :128-181) — global batch 32 * N, wall clock
  strong_scaling BASELINE config 2 as written: the SAME path with global batch 32 (32 / N images per GPU)
  stock_torch_fp16  the comparator a maintainer would otherwise run on this GPU: the same graph in stock PyTorch fp16
                 (cuDNN convs, cuBLAS linears, SDPA attention), same batch, device-timed.  Not part of the product.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
EXT = os.path.join(ROOT, "stable-diffusion-webui-distributed_b200")
for p in (ROOT, EXT, os.path.join(ROOT, "tests", "hoststub")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

STEPS_DDIM = 20     # sampler steps (the name is historical: --model sdxl runs 30 Euler a steps)
SAMPLER = "DDIM"
CFG_SCALE = 7.0
HW = 64  # 512 x 512 images
DENOISE = 0.75   # img2img (BASELINE config 3; SURVEY §8d)

# algorithmic FLOPs (SURVEY.md App. D / BASELINE.md §3), TFLOP
UNET_TFLOP_PER_SAMPLE_EVAL = 0.8033
VAE_TFLOP_PER_IMAGE = 2.5145
VAE_ENC_TFLOP_PER_IMAGE = 1.1167
CLIP_TFLOP_PER_SEQ = 0.0133
ATTN_TFLOP_PER_SAMPLE_EVAL = 0.1225
MODEL_NAME, DTYPE = "SD1.5", "fp16"


def select_model(name: str):
    """BASELINE config 4: SDXL-base txt2img 1024x1024, bf16, 30 Euler a steps (SURVEY App. D FLOP model)"""
    global STEPS_DDIM, SAMPLER, HW, UNET_TFLOP_PER_SAMPLE_EVAL, VAE_TFLOP_PER_IMAGE, VAE_ENC_TFLOP_PER_IMAGE, CLIP_TFLOP_PER_SEQ
    global MODEL_NAME, DTYPE
    if name in ("sdxl", "tinyxl"):
        STEPS_DDIM, SAMPLER, HW = 30, "Euler a", 128
        UNET_TFLOP_PER_SAMPLE_EVAL, VAE_TFLOP_PER_IMAGE, VAE_ENC_TFLOP_PER_IMAGE = 6.7612, 10.4704, 4.65
        CLIP_TFLOP_PER_SEQ = 0.0133 + 0.107      # CLIP-L + OpenCLIP bigG text towers (694 M parameters x 77 tokens x 2)
        MODEL_NAME, DTYPE = "SDXL-base", "bf16"
MUFU_EXP_PER_CLK_SM = 16      # MUFU.EX2 per clock and SM (B300_MICROARCH.md; tools/xu_probe.cu measured 4.47 T/s at 1.9 GHz)
NUM_SMS = 148


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"tflops_burst": d["bf16_tflops"], "tflops_sustained": d["bf16_tflops_sustained"], "hbm_gbs": d["hbm_gbs"],
                "source": "measured"}
    return {"tflops_burst": 1590.0, "tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms",
                                          "200", "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                                         text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=3)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def usable_cpus() -> int:
    """host cores this process may really use: affinity mask, capped by the cgroup CPU quota (containers often
    advertise every core of the host in os.cpu_count() while being limited to a few)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, q // per))
        except (OSError, ValueError, IndexError):
            continue
    return max(1, n)


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ================================================================================================ CPU arms (oracle)
# The ONLY part of this file that touches oracle/: the reference's numeric path on host cores, as a checker-grade
# baseline.  None of it is reachable from the GPU arm's timed regions.
def cpu_bounded_sample(n_evals: int, threads: int, unet_reps: int = 1):
    """`cpu_baseline` of the GPU arm's line: a BOUNDED sample (one CFG UNet evaluation of one image + one VAE decode +
    two CLIP encodes, ~10 s), composed to one image.  An estimate by construction; the measured whole request is the
    reference arm (--impl reference)."""
    from b200sd import config as C, synth
    from oracle import sd_oracle as O
    torch.set_num_threads(threads)
    cfgs = (C.SD15_UNET, C.SD15_VAE, C.SD15_CLIP)
    sd = synth.make_state_dict(*cfgs, seed=0)
    tok = O.random_prompt_tokens(1)
    neg = O.empty_prompt_tokens(1)
    with torch.no_grad():
        t0 = time.perf_counter()
        cond = O.clip_text_encode(sd, cfgs[2], tok)
        unc = O.clip_text_encode(sd, cfgs[2], neg)
        t_clip = time.perf_counter() - t0
        x = O.per_image_noise(1000, 1, (4, HW, HW))
        ts = []
        for _ in range(unet_reps):
            t0 = time.perf_counter()
            O.cfg_eps(lambda a, t, c: O.unet_forward(sd, cfgs[0], a, t, c), x, 651, cond, unc, CFG_SCALE)
            ts.append(time.perf_counter() - t0)
        t_unet = min(ts)
        t0 = time.perf_counter()
        O.to_uint8(O.vae_decode(sd, cfgs[1], x))
        t_vae = time.perf_counter() - t0
    sec_per_image = n_evals * t_unet + t_vae + t_clip
    return {"value": 1.0 / sec_per_image, "unit": "images/s", "cores": threads, "kind": "port",
            "sample": f"ESTIMATE composed from a bounded sample: {unet_reps} CFG UNet eval(s) of 1 image ({t_unet:.2f}s) x {n_evals} + "
                      f"1 VAE decode ({t_vae:.2f}s) + 2 CLIP encodes ({t_clip:.2f}s), fp32 torch on {threads} host threads",
            "sec_per_image": sec_per_image}


class OracleCPUEngine:
    """'stock sdwui on CPU' stand-in (sdwui itself is not installable offline): the fp32 oracle behind the call surface
    LocalGPUWorker / server.sdapi use, so the HTTP-dispatch path can run end to end on host cores."""

    def __init__(self, threads: int, size: str = "sd15"):
        from b200sd import factory
        self.cfgs = factory.configs(size)
        self.sd = factory.state_dict(size)
        self.unet_cfg, self.vae_cfg, self.clip_cfg = self.cfgs
        self.interrupted = False
        self.variation = (None, 0.0)
        self.threads = threads
        self.last_unet_evals = 0

    def txt2img(self, tok, neg, seed, steps=20, cfg_scale=7.0, height=512, width=512, sampler="DDIM", scheduler=None):
        from oracle import sd_oracle as O
        torch.set_num_threads(self.threads)
        with torch.no_grad():
            u8, _, _ = O.txt2img(self.sd, *self.cfgs, tok, neg, seed=seed, steps=steps, cfg_scale=cfg_scale, height=height,
                                 width=width, sampler="DDIM")
        return u8


def serve_cpu_oracle(port: int, threads: int, size: str):
    """child process of the reference arm: an sdwui-API worker (server/sdapi.py) whose executor is the CPU oracle"""
    import logging
    import uvicorn
    from scripts.spartan import pmodels, shared as sh
    from server.sdapi import create_app
    logging.getLogger("distributed").setLevel(logging.ERROR)
    sh.benchmark_payload = pmodels.Benchmark_Payload()
    eng = OracleCPUEngine(threads, size)
    uvicorn.run(create_app(lambda device: eng, [0]), host="127.0.0.1", port=port, log_level="error")


def _free_port() -> int:
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def reference_http_dispatch_arm(size: str = "sd15", steps: int = STEPS_DDIM, hw: int = HW, max_requests: int = 1):
    """BASELINE config 1: txt2img 512x512 batch 2, master + 1 worker, both on host cores, through the extension's HTTP
    dispatch path: DistributedScript.before_process -> World.optimize_jobs -> Worker.request (requests.post to
    /sdapi/v1/txt2img, reference worker.py:423-448) -> postprocess_batch_list -> postprocess.  The master generates its
    share in-process while the worker's HTTP call is in flight (one thread per job, distributed.py:316-318).
    The dispatcher is this repo's mirror of the reference's (pinned to it bit for bit by tests/test_scheduler_parity.py;
    /root/reference itself does not travel to the GPU box — profiles/r02_reference_http_dispatch_container.json holds the
    same run driven by the UNMODIFIED reference dispatcher in the build container); the workers are the fp32 oracle.
    A whole request is timed for real (no extrapolation): wall clock before_process entry -> postprocess exit."""
    import logging
    import requests
    import modules.processing as processing
    import modules.scripts as mscripts
    from scripts.distributed import DistributedScript
    from scripts.spartan import pmodels, shared as sh
    from scripts.spartan.world import World
    logging.getLogger("distributed").setLevel(logging.ERROR)
    cores = usable_cpus()
    threads = max(1, cores // 2)
    port = _free_port()
    child = subprocess.Popen([sys.executable, os.path.abspath(__file__), "--serve-cpu-oracle", str(port), "--threads", str(threads),
                              "--model", size], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    try:
        for _ in range(600):
            try:
                if requests.get(f"http://127.0.0.1:{port}/sdapi/v1/memory", timeout=1).status_code == 200:
                    break
            except requests.RequestException:
                time.sleep(0.2)
        else:
            raise RuntimeError("the CPU worker did not come up")
        master_engine = OracleCPUEngine(threads, size)
        from b200sd.factory import synthetic_tokens

        def master_generator(p, n):
            v = master_engine.clip_cfg.vocab
            tok = synthetic_tokens([p.prompt] * p.batch_size, v)
            neg = synthetic_tokens([p.negative_prompt] * p.batch_size, v)
            u8 = master_engine.txt2img(tok, neg, p.seeds[0], steps=p.steps, cfg_scale=p.cfg_scale, height=p.height, width=p.width)
            return [u8[i].permute(2, 0, 1).float() / 255.0 for i in range(u8.shape[0])]

        processing.MASTER_GENERATOR = master_generator
        sh.benchmark_payload = pmodels.Benchmark_Payload()
        w = World(verify_remotes=False)
        DistributedScript.world = w
        w.master().avg_ipm, w.master().benchmarked = 1.0, True
        wk = w.add_worker(address="127.0.0.1", port=port, label="cpu-worker", avg_ipm=1.0, master=False, verify_remotes=False)
        wk.benchmarked = True
        w.benchmark = lambda *a, **k: None     # equal speeds set above: batch 2 -> 1 image each
        w.job_timeout = 3600
        script = DistributedScript()
        script.args_from = script.args_to = 0
        times, n_images = [], 0
        for it in range(max_requests):
            p = processing.StableDiffusionProcessingTxt2Img(
                prompt="a synthetic benchmark prompt", negative_prompt="", seed=1000, subseed=1, subseed_strength=0, batch_size=2,
                n_iter=1, steps=steps, width=hw * 8, height=hw * 8, sampler_name="DDIM", cfg_scale=CFG_SCALE,
                scripts=mscripts.ScriptRunner([script]), script_args=[])
            t0 = time.perf_counter()
            out = processing.process_images(p)
            times.append(time.perf_counter() - t0)
            n_images = len(out.images)
            if n_images != 2:
                raise RuntimeError(f"HTTP dispatch returned {n_images} images instead of 2")
    finally:
        child.terminate()
        try:
            child.wait(timeout=5)
        except subprocess.TimeoutExpired:
            child.kill()
    best = min(times)
    return {"value": n_images / best, "unit": "images/s", "cores": cores, "kind": "port", "sec_per_request": best,
            "requests_timed": len(times),
            "sample": f"{len(times)} whole request(s), measured not composed: txt2img {hw * 8}x{hw * 8} batch 2, {steps} DDIM timesteps, "
                      f"master + 1 HTTP worker (server/sdapi.py over loopback), each the fp32 oracle on {threads} of {cores} host "
                      f"threads, wall clock before_process -> postprocess = {best:.1f}s"}


# ================================================================================================ GPU arm helpers
def stock_torch_fp16(b: int, n_evals: int, dev: str, size: str = "sd15"):
    """Comparator (not the product): the SAME graph in stock PyTorch on this GPU — fp16 weights/activations, cuDNN
    convolutions, cuBLAS linears, F.scaled_dot_product_attention, fp32 GroupNorm/LayerNorm statistics as ldm runs them —
    one whole request of the bench batch, device-timed.  The graph is the oracle's (restating ldm is restating it);
    what is measured here is the libraries, so the oracle-as-checker rule is not in play."""
    from b200sd import factory
    from oracle import sd_oracle as O
    cfgs = factory.configs(size)
    sd = {k: v.to(dev, torch.float16) for k, v in factory.state_dict(size).items()}
    g = torch.Generator().manual_seed(1234)
    vocab = cfgs[2].vocab
    tokens = torch.cat([torch.full((b, 1), vocab - 2), torch.randint(0, vocab - 3, (b, 75), generator=g),
                        torch.full((b, 1), vocab - 1)], dim=1).to(dev)
    neg = torch.full((b, 77), vocab - 1)
    neg[:, 0] = vocab - 2
    neg = neg.to(dev)
    x_T = O.per_image_noise(1000, b, (4, HW, HW)).to(dev, torch.float16)
    O.USE_SDPA = True
    unet = lambda a, t, c: O.unet_forward(sd, cfgs[0], a, t, c)  # noqa: E731

    def request():
        with torch.no_grad():
            cond, unc = O.clip_text_encode(sd, cfgs[2], tokens), O.clip_text_encode(sd, cfgs[2], neg)
            z = O.sample_ddim(unet, x_T, cond, unc, STEPS_DDIM, CFG_SCALE)
            outs = [O.to_uint8(O.vae_decode(sd, cfgs[1], z[i:i + 8] / cfgs[1].scale_factor)) for i in range(0, b, 8)]
        return torch.cat(outs)

    try:
        request()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 2
        e0.record()
        for _ in range(reps):
            request()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        res = {"value": b / (ms / 1000.0), "unit": "images/s", "ms_per_request": ms, "batch": b, "unet_evals": n_evals,
               "what": "stock PyTorch fp16 (cuDNN / cuBLAS / SDPA), eager, same graph, same batch, same GPU, device-timed; "
                       "comparator only", "torch": torch.__version__}
    except Exception as e:   # a comparator must never take the bench line down
        res = {"value": None, "error": f"{type(e).__name__}: {str(e)[:200]}"}
    finally:
        O.USE_SDPA = False
        del sd
        torch.cuda.empty_cache()
    return res


def plugin_world(engine_factory, devices, thin=True):
    """a fresh World holding one LocalGPUWorker per device (thin-client master), and a DistributedScript bound to it"""
    import logging
    from scripts.distributed import DistributedScript
    from scripts.spartan import pmodels, shared as sh
    from scripts.spartan.world import World
    logging.getLogger("distributed").setLevel(logging.ERROR)
    sh.benchmark_payload = pmodels.Benchmark_Payload()
    w = World(verify_remotes=False)
    DistributedScript.world = w
    for wk in w.add_local_gpus(engine_factory, devices=list(devices), avg_ipm=600.0):
        wk.benchmarked = True
    w.thin_client_mode = thin
    w.benchmark = lambda *a, **k: None      # speeds are set above; do not re-benchmark inside the timed region
    script = DistributedScript()
    script.args_from = script.args_to = 0
    return w, script


def plugin_request(script, batch, tokens, seed0, workload, init_images=None):
    import modules.processing as processing
    import modules.scripts as mscripts
    kw = dict(prompt="synthetic", negative_prompt="", seed=seed0, subseed=1, subseed_strength=0, batch_size=batch, n_iter=1,
              steps=STEPS_DDIM, width=HW * 8, height=HW * 8, sampler_name=SAMPLER, cfg_scale=CFG_SCALE,
              scripts=mscripts.ScriptRunner([script]), script_args=[])
    if workload == "img2img":
        p = processing.StableDiffusionProcessingImg2Img(init_images=init_images, denoising_strength=DENOISE, **kw)
    else:
        p = processing.StableDiffusionProcessingTxt2Img(**kw)
    p.prompt_tokens = tokens                # host token ids ride along in the payload (p.__dict__); a tensor: the per-job
                                            # deepcopy of the payload (reference distributed.py:288-290) is then a memcpy
    return processing.process_images(p)


def synthetic_inputs(eng, b, rank):
    from b200sd import engine as E
    vocab = eng.clip_cfg.vocab
    g = torch.Generator().manual_seed(1234 + rank)
    tokens = torch.cat([torch.full((b, 1), vocab - 2), torch.randint(0, vocab - 3, (b, 75), generator=g),
                        torch.full((b, 1), vocab - 1)], dim=1)
    neg = torch.full((b, 77), vocab - 1)
    neg[:, 0] = vocab - 2
    seed0 = 1000 + rank * b   # global image index -> seed (reference: seed + images owned by earlier jobs)
    x_T = E.per_image_noise(seed0, b, (4, HW, HW))[0]
    g2 = torch.Generator().manual_seed(4321 + rank)
    init_u8 = torch.randint(0, 256, (b, HW * 8, HW * 8, 3), generator=g2, dtype=torch.uint8)   # SURVEY §8d img2img init
    return tokens, neg, seed0, x_T, init_u8


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, images):
    """images [n, H, W, 3] uint8 -> out_dir/images.npy float32 (values 0..255) and out_dir/images_index.npy float64 (their
    indices in the batch).  Whole images are kept, as many as fit DUMP_BYTES, chosen by a fixed seed, so that two builds
    run with the same arguments write the same images and can be compared value for value."""
    import numpy as np
    n = images.shape[0]
    per_image = images[0].numel() * 4 + 8
    keep = min(n, (DUMP_BYTES - 1024) // per_image)   # 1024: the two .npy headers
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "images.npy"), images.cpu()[idx].float().numpy())
    np.save(os.path.join(out_dir, "images_index.npy"), idx.double().numpy())


def make_step(eng, workload, b, tokens_d, neg_d, x_T_d, init_d, seed0, world, gather):
    """one request with its inputs already on the device: conditioning, sampling, VAE decode (+ the all-gather)"""
    from b200sd import engine as E
    px = HW * 8
    pr = eng.program(SAMPLER, None, STEPS_DDIM, denoise=DENOISE if workload == "img2img" else None)
    draws = None
    if pr.draws:   # Euler a (SDXL config): the per-image ancestral draws of this rank's seeds, resident like x_T
        draws = E.per_image_noise(seed0, b, (4, HW, HW), 1 + pr.draws)[1:].to(x_T_d.device)

    def step():
        cond, unc = eng._conds(tokens_d, neg_d, px, px)
        init = eng.encode(init_d) if workload == "img2img" else None
        lat = eng.run_program(cond, unc, pr.start(x_T_d, init), pr, CFG_SCALE, noises=draws)
        u8 = eng.decode(lat, HW, HW)
        if world > 1:
            u8 = gather(u8, [b] * world)
        return u8

    return step


def timed_device(eng, step, steps, warmup, barrier, rank, local, world, dev):
    """W >= 3 untimed requests, then exactly K timed ones between barrier + synchronize on both sides; CUDA events, max
    over ranks.  Returns (ms, clocks during the timed region, b200sd kernels launched inside it, the last timed step's
    images)."""
    import torch.distributed as dist
    from b200sd import ops
    for _ in range(max(3, warmup)):
        step()
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    l0 = ops.LAUNCHES + eng.graph_replayed_launches
    e0.record()
    for _ in range(steps):
        out = step()
    e1.record()
    barrier()
    launches = ops.LAUNCHES + eng.graph_replayed_launches - l0
    ms = e0.elapsed_time(e1)
    clk = clocks.stop() if rank == 0 else None
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), clk, launches, out


# ================================================================================================ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--per-gpu-batch", type=int, default=0, help="default: 32 (SD1.5), 16 (SDXL): BASELINE's batch on one GPU")
    ap.add_argument("--model", default="sd15", choices=["sd15", "tiny", "sdxl", "tinyxl"])
    ap.add_argument("--workload", default="txt2img", choices=["txt2img", "img2img"])
    ap.add_argument("--sweep", default=None, help="comma-separated per-GPU batches (BASELINE config 5): one JSON line with a list")
    ap.add_argument("--sweep-out", default=None, help="also run the sweep of --sweep-batches after the main measurement -> JSON file")
    ap.add_argument("--sweep-batches", default="1,2,4,8,16,64")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-world", action="store_true")
    ap.add_argument("--no-stock", action="store_true")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the images of the last timed step to DIR/images.npy (float32; a seeded sample of whole "
                         "images when the batch exceeds 64 MB) and their batch indices to DIR/images_index.npy")
    ap.add_argument("--serve-cpu-oracle", type=int, default=None, help=argparse.SUPPRESS)
    ap.add_argument("--threads", type=int, default=0, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.sweep or args.impl == "reference"):
        ap.error("--dump-outputs applies to the main measurement of --impl b200, not to --sweep or --impl reference")
    if args.serve_cpu_oracle is not None:
        return serve_cpu_oracle(args.serve_cpu_oracle, args.threads or usable_cpus(), args.model)
    rank, world, local = dist_env()
    select_model(args.model)
    xl = args.model in ("sdxl", "tinyxl")
    args.per_gpu_batch = args.per_gpu_batch or (16 if xl else 32)
    img2img = args.workload == "img2img"
    if xl and img2img:
        raise SystemExit("--workload img2img is BASELINE config 3 (SD1.5)")
    n_evals = STEPS_DDIM if xl else ((int(DENOISE * STEPS_DDIM) - 1) if img2img else STEPS_DDIM - 1)
    px = HW * 8
    workload = (f"{MODEL_NAME} {args.workload} {px}x{px} {DTYPE}, {STEPS_DDIM} {SAMPLER} steps"
                + (f", denoising strength {DENOISE}: VAE encode + {n_evals}" if img2img else f" = {n_evals}")
                + f" CFG UNet evaluations + VAE decode, per-GPU batch {args.per_gpu_batch}, batch-sharded by image index, "
                  f"synthetic seeded weights, random-token prompts")
    config = {"workload": workload, "per_gpu_batch": args.per_gpu_batch, "global_batch": args.per_gpu_batch * world,
              "resolution": f"{px}x{px}", "sampler": SAMPLER, "timesteps": STEPS_DDIM, "unet_evals": n_evals,
              "cfg_scale": CFG_SCALE, "parallelism": f"dp{world} (batch index sharding, one all-gather at the end)",
              "l2": "every step streams far more than the 126 MB L2 (activations of one UNet eval at batch 64 exceed 10 GB)"}

    if args.impl == "reference":
        if rank != 0:
            return
        t0 = time.perf_counter()
        r = reference_http_dispatch_arm(args.model, max_requests=1)
        line = {"impl": "reference", "metric": "images/sec SD1.5 512x512 txt2img", "value": r["value"],
                "unit": "images/s", "n_gpus": args.gpus, "gpus_used": 0,
                # one whole request is timed for real (minutes on host cores): the requested K / W are recorded, not honoured
                "steps": r["requests_timed"], "warmup": 0, "steps_requested": args.steps, "warmup_requested": args.warmup,
                "ms_per_step": r["sec_per_request"] * 1000.0, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
                "config": config,
                "reference_workload": "BASELINE config 1: txt2img 512x512 batch 2, 20 DDIM timesteps, master + 1 HTTP worker on host "
                                      "cores — images/s of the same metric on the reference's own dispatch path",
                "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": r["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "wall_s": time.perf_counter() - t0}
        print(json.dumps(line))
        return

    import torch.distributed as dist
    from b200sd import factory, ops
    from b200sd.sharding import all_gather_images
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    cpu_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
        cpu_group = dist.new_group(backend="gloo")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    eng = factory.default_engine_factory(dev, args.model)

    # ---------------- BASELINE config 5: per-GPU batch sweep (device-timed whole requests, weak scaling per batch)
    def run_sweep(batches):
        rows = []
        for bb in batches:
            tk, ng, sd0, xt, iu8 = synthetic_inputs(eng, bb, rank)
            step = make_step(eng, args.workload, bb, tk.to(dev), ng.to(dev), xt.to(dev), iu8.to(dev), sd0, world,
                             all_gather_images)
            ms, ck, _, _ = timed_device(eng, step, args.steps, args.warmup, barrier, rank, local, world, dev)
            rows.append({"per_gpu_batch": bb, "global_batch": bb * world, "value": world * bb * args.steps / (ms / 1000.0),
                         "ms_per_step": ms / args.steps, "clocks": ck})
            eng.plans.pop((bb, HW, HW), None)
            torch.cuda.empty_cache()
        tfl = 2 * n_evals * UNET_TFLOP_PER_SAMPLE_EVAL + VAE_TFLOP_PER_IMAGE + 2 * CLIP_TFLOP_PER_SEQ
        for r in rows:
            r["step_roofline_frac"] = r["value"] * tfl / world / peaks()["tflops_sustained"]
        return {"metric": f"images/sec {MODEL_NAME} {px}x{px} {args.workload}", "unit": "images/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(3, args.warmup), "scaling": "weak per batch (per-GPU batch fixed, N ranks)",
                "dtype": DTYPE, "workload": args.workload, "pdl": os.environ.get("B200SD_PDL", "default (small grids only)"),
                "sweep": rows}

    if args.sweep:
        res = run_sweep([int(v) for v in args.sweep.split(",")])
        if rank == 0:
            print(json.dumps(res))
        if world > 1:
            dist.destroy_process_group()
        return

    b = args.per_gpu_batch
    tokens, neg, seed0, x_T, init_u8 = synthetic_inputs(eng, b, rank)
    step_device = make_step(eng, args.workload, b, tokens.to(dev), neg.to(dev), x_T.to(dev), init_u8.to(dev), seed0, world,
                            all_gather_images)
    elapsed_ms, clk, gpu_launches, images = timed_device(eng, step_device, args.steps, args.warmup, barrier, rank, local,
                                                         world, dev)
    value = world * b * args.steps / (elapsed_ms / 1000.0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, images)

    # ---------------- e2e through the plugin surface (host buffers, H2D + D2H inside the timed region), one world per rank
    e2e = None
    init_pil = None
    if img2img:
        from PIL import Image
        init_pil = [Image.fromarray(init_u8[i].numpy()) for i in range(b)]
    if not args.no_e2e:
        w, script = plugin_world(lambda d: eng, [local])
        for _ in range(2):
            out = plugin_request(script, b, tokens, seed0, args.workload, init_pil)
        assert len(out.images) == b, len(out.images)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            plugin_request(script, b, tokens, seed0, args.workload, init_pil)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        e2e = {"value": world * b * args.steps / dt, "unit": "images/s",
               "h2d_bytes_per_step": int(tokens.numel() * 8 + neg.numel() * 8 + x_T.numel() * 4
                                         + (init_u8.numel() if img2img else 0)),
               # the uint8 images and their CHW float copies for sdwui's postprocess hooks (made on the device)
               "d2h_bytes_per_step": int(b * HW * 8 * HW * 8 * 3 * (1 + 4)),
               "path": "hoststub process_images -> DistributedScript.before_process -> LocalGPUWorker.request -> "
                       "postprocess_batch_list -> postprocess (thin-client world, 1 local GPU per rank)"}

    if args.sweep_out:
        res = run_sweep([int(v) for v in args.sweep_batches.split(",")])
        res["sweep"].append({"per_gpu_batch": b, "global_batch": b * world, "value": value, "ms_per_step": elapsed_ms / args.steps,
                             "clocks": clk, "note": "the main measurement of this run"})
        if rank == 0:
            with open(args.sweep_out, "w") as f:
                json.dump(res, f)

    # ---------------- one process, ONE World over all N GPUs (rank 0 drives; the other ranks idle at the barrier)
    world_e2e = strong = None
    if not args.no_world and not args.no_e2e:
        # the other ranks wait on a HOST barrier (gloo): an NCCL barrier would park a spinning kernel on their GPUs, which
        # rank 0 is about to drive from this process
        barrier()
        if rank == 0:
            try:
                world_e2e, strong = world_level(args, world, b, tokens, seed0, init_pil, eng, local)
            except Exception as e:   # a secondary measurement must never take the headline line down
                world_e2e = strong = {"value": None, "error": f"{type(e).__name__}: {str(e)[:300]}"}
        if world > 1:
            dist.barrier(group=cpu_group)
        barrier()

    # ---------------- roofline of the dominant kernel: per-launch CUDA-event timing of one eager UNet evaluation
    try:
        roof, roof_attn, breakdown = kernel_rooflines(eng, b, peaks(), clk)
    except Exception as e:
        roof = roof_attn = {"frac": None, "error": f"{type(e).__name__}: {str(e)[:300]}"}
        breakdown = None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    tflop_per_image = 2 * n_evals * UNET_TFLOP_PER_SAMPLE_EVAL + VAE_TFLOP_PER_IMAGE + 2 * CLIP_TFLOP_PER_SEQ \
        + (VAE_ENC_TFLOP_PER_IMAGE if img2img else 0.0)
    line = {
        "metric": f"images/sec {MODEL_NAME} {px}x{px} {args.workload}", "value": value, "unit": "images/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": elapsed_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
        "config": config, "clocks": clk, "gpu_launches": int(gpu_launches), "e2e": e2e,
        "world_e2e": world_e2e, "strong_scaling": strong,
        "roofline": roof, "roofline_attention": roof_attn, "unet_eval_breakdown_ms": breakdown,
        "step_roofline": {"bound": "tensor", "achieved": value * tflop_per_image / world, "peak": pk["tflops_sustained"],
                          "unit": "TFLOP/s", "frac": value * tflop_per_image / world / pk["tflops_sustained"],
                          "tflop_per_image": tflop_per_image, "peak_source": pk["source"] + " (sustained)"},
    }
    if world == 1 and not args.no_stock and args.model == "sd15" and not img2img:
        eng.plans.clear()
        torch.cuda.empty_cache()
        line["stock_torch_fp16"] = stock_torch_fp16(b, n_evals, dev, args.model)
        if line["stock_torch_fp16"].get("value"):
            line["stock_torch_fp16"]["speedup_of_this_repo"] = value / line["stock_torch_fp16"]["value"]
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = {k: v for k, v in cpu_bounded_sample(n_evals, usable_cpus()).items()
                                if k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def world_level(args, world, b, tokens, seed0, init_pil, eng0, local0):
    """rank 0: ONE DistributedScript, a LocalGPUWorker for every GPU of the job, one request.  Under torchrun the other
    ranks keep their own engines on their GPUs (idle at a barrier meanwhile); this process builds one more engine per
    remote device — the in-process design of the north star."""
    from b200sd import factory
    devs = list(range(world))
    engines = {f"cuda:{local0}": eng0}

    def fac(device):
        if device not in engines:
            engines[device] = factory.default_engine_factory(device, args.model)
        return engines[device]

    w, script = plugin_world(fac, devs)
    res = []
    for gb in (b * world, b):   # weak (32 per GPU) and BASELINE config 2 as written (32 in total)
        if gb % world:
            res.append(None)
            continue
        g = torch.Generator().manual_seed(99)
        toks = tokens[:1].expand(gb, -1).contiguous() if gb > tokens.shape[0] else tokens[:gb]
        imgs = None if init_pil is None else [init_pil[i % len(init_pil)] for i in range(gb)]
        for _ in range(2):
            out = plugin_request(script, gb, toks, seed0, args.workload, imgs)
        # the warm-up requests built plans and captured graphs on the devices this process had not used yet: their ETA
        # errors say nothing about steady state, and the scheduler would read them as lag (complementary jobs, bonus images)
        for wk in w.get_workers():
            wk.eta_percent_error = []
        for d in devs:
            torch.cuda.synchronize(d)
        reps = max(2, min(args.steps, 5))
        n_img = 0
        t0 = time.perf_counter()
        for _ in range(reps):
            out = plugin_request(script, gb, toks, seed0, args.workload, imgs)
            n_img += len(out.images)
        for d in devs:
            torch.cuda.synchronize(d)
        dt = (time.perf_counter() - t0) / reps
        res.append({"value": n_img / reps / dt, "unit": "images/s", "global_batch": gb, "per_gpu_batch": gb // world, "n_gpus": world,
                    "images_returned_per_request": n_img / reps, "ms_per_request": dt * 1000.0, "requests_timed": reps,
                    "jobs": [j.batch_size for j in w.jobs if j.batch_size > 0],
                    "path": "ONE process: process_images -> DistributedScript.before_process -> World.optimize_jobs -> one "
                            "thread per LocalGPUWorker job -> collector (tensors lane) -> postprocess; wall clock, host "
                            "buffers in and out"})
    for k in [k for k in engines if k != f"cuda:{local0}"]:
        engines.pop(k).release()
        factory.evict(k)
    return res[0], res[1]


def kernel_rooflines(eng, b, pk, clk):
    """Per-launch CUDA-event durations of every kernel class in ONE eager UNet evaluation (same shapes as the timed
    region).  roofline = the dominant kernel (gemm_conv_tc_kernel: all convs and linears), ALGORITHMIC FLOPs (unpadded
    shapes: zero-padded head columns and latent channels are layout, not work) summed over its launches / summed
    duration, against the measured sustained bf16 tensor peak."""
    from b200sd import ops
    plan = eng.plan(b, HW, HW)
    ops.select_step(plan.table, plan.step * 0, plan.unet.cur_bias)
    torch.cuda.synchronize()
    recs = []
    exps = [0.0]   # exponentials of all attention launches (one per S element)
    padded = [0.0]
    for (fn, a, k), algo in zip(plan.unet.ops, plan.unet.op_flops):
        name = getattr(fn, "__name__", "op")
        name = "groupnorm" if name == "<lambda>" else name
        flop = 0.0
        if name in ("linear", "conv2d"):
            m = (a[0].numel() // a[0].shape[-1]) if name == "linear" else (a[2].numel() // a[2].shape[-1])
            packed = 2.0 * m * a[1].shape[0] * a[1].shape[1]
            flop = packed if algo is None else algo
            padded[0] += packed
        elif name == "attention":
            bq, sq, skv, heads, d = a[0].shape[0], a[0].shape[1], a[1].shape[1], a[4], a[5]
            flop = 4.0 * bq * heads * sq * skv * d
            exps[0] += float(bq) * heads * sq * skv
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn(*a, **k)
        e1.record()
        recs.append((name, flop, e0, e1))
    torch.cuda.synchronize()
    agg = {}
    for name, flop, e0, e1 in recs:
        d = agg.setdefault(name, [0, 0.0, 0.0])
        d[0] += 1; d[1] += e0.elapsed_time(e1); d[2] += flop
    tc = [agg.get("linear", [0, 0, 0]), agg.get("conv2d", [0, 0, 0])]
    n_l, ms, fl = (sum(x[i] for x in tc) for i in range(3))
    peak = pk["tflops_sustained"]
    traffic = traffic_src = None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic = tj.get("gemm_conv_tc_kernel_dram_bytes_per_launch")
        traffic_src = tj.get("source", "ncu capture committed under profiles/ (not measured in this run)")
    roof = {"kernel": "gemm_conv_tc_kernel (all conv2d + linear launches of one UNet evaluation)", "bound": "tensor",
            "achieved": fl / (ms * 1e-3) / 1e12, "peak": peak, "unit": "TFLOP/s", "frac": fl / (ms * 1e-3) / 1e12 / peak,
            "traffic": traffic, "traffic_source": traffic_src, "launches": n_l, "avg_launch_us": ms * 1e3 / max(1, n_l),
            "algorithmic_flop_per_launch": fl / max(1, n_l),
            "flop_accounting": f"unpadded shapes: {fl / 1e12:.2f} TFLOP per evaluation at UNet batch {2 * b} "
                               f"({fl / 1e12 / (2 * b):.4f} per sample; SURVEY §8d 0.6772); the packed operands execute "
                               f"{padded[0] / 1e12:.2f}",
            "by_op": {"linear": {"ms": tc[0][1], "tflops": tc[0][2] / max(tc[0][1], 1e-9) / 1e9},
                      "conv2d": {"ms": tc[1][1], "tflops": tc[1][2] / max(tc[1][1], 1e-9) / 1e9}},
            "peak_source": pk["source"] + " sustained bf16 cuBLAS"}
    at = agg.get("attention", [0, 1e-9, 0])
    sm_mhz = (clk or {}).get("sm_mhz") or 1965.0
    exp_peak_run = NUM_SMS * MUFU_EXP_PER_CLK_SM * sm_mhz * 1e6 / 1e12
    exp_ach = exps[0] / (at[1] * 1e-3) / 1e12
    roof_attn = {"kernel": "attention_tc_kernel", "bound": "tensor", "achieved": at[2] / (at[1] * 1e-3) / 1e12, "peak": peak,
                 "unit": "TFLOP/s", "frac": at[2] / (at[1] * 1e-3) / 1e12 / peak, "launches": at[0], "ms": at[1],
                 "note": "QK^T + PV FLOPs; d=40 heads make this kernel exp-throughput (MUFU) bound, see DESIGN.md",
                 # the pipe that actually bounds it: one MUFU.EX2 per S element, 16 per clock and SM
                 "exp_rate": {"achieved": exp_ach, "unit": "T exp/s",
                              "peak_at_run_clock": exp_peak_run, "frac_at_run_clock": exp_ach / exp_peak_run,
                              "peak_at_boost": 4.47, "frac_at_boost": exp_ach / 4.47,
                              "peak_source": f"148 SMs x 16 MUFU.EX2/clk x {sm_mhz:.0f} MHz (median SM clock of the timed region); "
                                             "4.47 measured by tools/xu_probe.cu at boost"}}
    breakdown = {k: round(v[1], 3) for k, v in agg.items()}
    # HBM-bound kernel classes: algorithmic bytes (DESIGN.md section 4: GroupNorm 2 reads + 1 write of 45.1 M elements per
    # sample-evaluation, LayerNorm 1 read + 1 write of 34.7 M) over the summed CUDA-event durations, against the measured
    # copy bandwidth
    hbm = {}
    gn_fused = getattr(plan.unet, "gn_fused_elems", 0)
    for name, elems, nbytes in (("groupnorm", plan.unet.gn_elems, gn_fused * 4 + (plan.unet.gn_elems - gn_fused) * 6),
                                ("layernorm", plan.unet.ln_elems, plan.unet.ln_elems * 4)):
        if name in agg and agg[name][1] > 0:
            gbs = nbytes / (agg[name][1] * 1e-3) / 1e9
            hbm[name] = {"bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"],
                         "launches": agg[name][0], "algorithmic_bytes": nbytes, "elements": elems, "ms": agg[name][1]}
            if name == "groupnorm":   # bytes the kernels actually move: 1 read + 1 write through the one-pass kernel, 2 + 1 else
                hbm[name]["one_pass_elements"] = gn_fused
                hbm[name]["frac_at_4_bytes_per_element"] = elems * 4 / (agg[name][1] * 1e-3) / 1e9 / pk["hbm_gbs"]
    roof["hbm_kernels"] = hbm
    return roof, roof_attn, breakdown


if __name__ == "__main__":
    main()
