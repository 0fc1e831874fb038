#!/usr/bin/env python
"""Headline benchmark: 512x512 LCM 4-step images/sec (UNet + VAE) — BASELINE.json metric.

  python bench.py --gpus N --steps K --warmup W                 # the B200-native arm, config C2
  python bench.py --impl reference --gpus N --steps K ...        # the reference's CPU path (oracle port)
  python bench.py --config c3 | c5 ...                           # BASELINE configs C3 / C5 (same arms)
  python bench.py --pool-workers N                               # ONE process, WorkerPool with N GPU workers
  python bench.py ... --dump-outputs DIR                         # + what the last timed step computed, DIR/<name>.npy

Config C2 (default): a "step" is one pass of the hot path over one batch: 4 x (UNet forward + LCM
scheduler step) followed by the VAE decode of a batch of 16 images (at N GPUs each rank runs its own
batch of 16 = config C4's 128/8 shard, weak scaling, no data-path collective).
  value       images/s, inputs resident in HBM, one CUDA-graph replay per step, CUDA events, L2 flushed
  e2e         the same metric through the reference-facing plugin boundary: `GenerationJob`s ->
              `WorkerPool.submit_job` -> `B200Worker.run_batch` -> PNG bytes (reference
              `backends/worker_pool.py:84-88`, `backends/cuda_worker.py:201-239`), host in, host out; PNG files
              assembled on the device (B200_PNG=gpu), with `e2e.e2e_png_pil` = the same pool with the
              reference's PIL encoder
  e2e_engine  the engine-level figure (pinned host tensors -> `LCMPipelineB200.generate` -> host u8)
Config C3: the same at 768x768, 8 steps, batch 8.  Config C5: SDXL-base arch, 1024x1024, 30 steps, CFG 7.5,
ONE image over the N ranks (CFG halves x row strips, `patch_parallel.py`), strong scaling.
One JSON line is printed by rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from types import SimpleNamespace

# the benchmark runs from a built tree that may be read-only: it writes nothing there, byte code included
sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

UNIT = "images/s"
DUMP_BYTES_MAX = 64 * 10**6
# algorithmic GFLOP per sample (2*MAC), SURVEY.md §8(d) / BASELINE.md §3
CONFIGS = {
    "c2": dict(arch="sd15", size=512, lcm_steps=4, batch=16, gs=1.0, gflop_unet=803.27, gflop_vae=2514.52,
               metric="512x512 LCM 4-step images/sec (UNet+VAE)"),
    "c3": dict(arch="sd15", size=768, lcm_steps=8, batch=8, gs=1.0, gflop_unet=2148.12, gflop_vae=5754.30,
               metric="768x768 LCM 8-step images/sec (UNet+VAE)"),
    "c5": dict(arch="sdxl", size=1024, lcm_steps=30, batch=1, gs=7.5, gflop_unet=2 * 6761.24, gflop_vae=10470.39,
               metric="SDXL 1024x1024 30-step CFG 7.5 images/sec, one image over N GPUs (patch parallel)"),
}


def gflop_image(c):
    return c["lcm_steps"] * c["gflop_unet"] + c["gflop_vae"]


def workload_text(c, per_gpu=True):
    if c["arch"] == "sdxl":
        return (f"SDXL-base arch (random-init seed 0) {c['size']}x{c['size']}, {c['lcm_steps']} LCM steps, CFG {c['gs']}, "
                f"1 image sharded over the ranks (UNet x{c['lcm_steps']} x2 CFG + scheduler + VAE decode)")
    return (f"SD1.5-LCM arch (random-init seed 0) {c['size']}x{c['size']}, {c['lcm_steps']} LCM steps, guidance {c['gs']}, "
            f"batch {c['batch']} per GPU (UNet x{c['lcm_steps']} + scheduler + VAE decode)")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1386.3), d.get("bf16_tflops", 1632.4), d.get("hbm_gbs", 6535.7), "measured"
    return 1400.0, 1590.0, 6650.0, "fallback"


def dump_outputs(out_dir, **arrays):
    """Writes each device tensor as out_dir/<name>.npy in float32, so that two builds run with the same arguments
    (hence the same seeded inputs) can be compared output for output.  Above DUMP_BYTES_MAX in all, every array is
    cut to a fixed, seeded sample of its flattened elements: the same positions on every run."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: v.float().cpu().numpy() for k, v in arrays.items()}
    frac = min(1.0, (DUMP_BYTES_MAX - 4096) / (4 * sum(a.size for a in arrays.values())))
    for name, a in arrays.items():
        if frac < 1.0:
            keep = np.random.default_rng(0).choice(a.size, int(a.size * frac), replace=False)
            a = a.reshape(-1)[np.sort(keep)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle (fp32 CPU restatement of the diffusers path) on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_reference(c, threads: int):
    """-> (once, sample_text, extrapolated).  once() runs ONE bounded sample of the workload on the host
    cores and returns (seconds the sample took, seconds per image it stands for).
    SD1.5 configs: the sample IS one image of the batch — the full pass through
    `oracle.pipeline.run_pipeline` (all UNet forwards + scheduler steps + the full-size VAE decode), so
    seconds per image is measured, not extrapolated.  C5 (416 TFLOP per image, ~10 minutes of CPU) is the
    one extrapolated case: one CFG UNet forward (batch 2) + the full 1024^2 decode, image = 30 x UNet + decode."""
    import torch
    torch.set_num_threads(threads)
    if c["arch"] == "sd15":
        from oracle.pipeline import build_random_init, run_pipeline, synthetic_inputs
        unet, vae = build_random_init(seed=0)
        pe, lat, noise = synthetic_inputs(1, c["size"], c["size"], c["lcm_steps"])

        def once():
            t0 = time.perf_counter()
            run_pipeline(unet, vae, pe, lat, noise, c["lcm_steps"], c["gs"], tiling=False)
            dt = time.perf_counter() - t0
            return dt, dt
        txt = (f"1 image of the batch (config C1 geometry, B=1): the full oracle pass run_pipeline() = {c['lcm_steps']} UNet "
               f"forwards + scheduler steps + {c['size']}^2 VAE decode, fp32 torch CPU restatement of the diffusers path; "
               f"images/s = 1 / seconds per pass (measured, not extrapolated)")
        return once, txt, False
    from oracle.pipeline import build_random_init, sdxl_time_ids, synthetic_inputs
    from oracle.unet import UNetConfig
    from oracle.vae import VAEConfig
    unet, vae = build_random_init(UNetConfig.sdxl_base(), VAEConfig(scaling_factor=0.13025, sample_size=1024), seed=0)
    pe, lat, _ = synthetic_inputs(1, c["size"], c["size"], 2, ctx_dim=2048)
    pooled = torch.randn(1, 1280, generator=torch.Generator().manual_seed(2))
    tid = sdxl_time_ids(c["size"], c["size"], 2)

    def once():
        with torch.no_grad():
            t0 = time.perf_counter()
            unet(torch.cat([lat, lat]), torch.tensor(999), torch.cat([torch.zeros_like(pe), pe]), None,
                 text_embeds=torch.cat([torch.zeros_like(pooled), pooled]), time_ids=tid)
            t1 = time.perf_counter()
            vae(lat / vae.cfg.scaling_factor, tiling=False)
            t2 = time.perf_counter()
        return t2 - t0, c["lcm_steps"] * (t1 - t0) + (t2 - t1)
    txt = (f"EXTRAPOLATED: one CFG UNet forward (batch 2) + the {c['size']}^2 VAE decode of the fp32 CPU oracle; seconds per "
           f"image = {c['lcm_steps']} x t_unet + t_vae (a full image is ~416 TFLOP of CPU work)")
    return once, txt, True


def run_reference(args, c):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    once, txt, extrapolated = cpu_reference(c, threads)
    for _ in range(args.warmup):
        once()
    runs = [once() for _ in range(args.steps)]
    sample_s = [r[0] for r in runs]
    per_image = statistics.median(r[1] for r in runs)
    v = 1.0 / per_image
    print(json.dumps({
        "impl": "reference", "metric": c["metric"], "value": v, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(sample_s) / len(sample_s),
        "higher_is_better": True, "scaling": "strong" if c["arch"] == "sdxl" else "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text(c),
                   "note": "reference arm = fp32 CPU port (oracle/) of the reference's diffusers path on the host cores; "
                           "each step is one bounded sample of the workload (cpu_baseline.sample); value = median over "
                           "the steps", "extrapolated": extrapolated},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": txt,
                         "seconds_per_sample_median": statistics.median(sample_s)},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ------------------------------------------------------------------------------------------------
# plugin boundary: WorkerPool -> B200Worker -> PNG
# ------------------------------------------------------------------------------------------------
class _Modes:
    """The slice of the reference's ModeConfigManager the pool reads (`server/mode_config.py:202-265`)."""

    def __init__(self, root, model):
        self.config = SimpleNamespace(model_root=root)
        self._mode = SimpleNamespace(model=model, model_path=os.path.join(root, model), loras=[])

    def get_default_mode(self):
        return "bench"

    def get_mode(self, name):
        if name != "bench":
            raise KeyError(name)
        return self._mode


class _Registry:
    def get_used_vram(self):
        return 0

    def register_model(self, **kw):
        pass

    def unregister_model(self, name):
        pass


def bench_model_dir(c, rank, barrier):
    """Random-init diffusers-layout model directory the worker loads (`MODEL_ROOT/MODEL`): written once
    per box by rank 0."""
    from dreamlab_b200 import synthetic as syn
    root = os.environ.get("B200_BENCH_MODEL_ROOT", os.path.join(tempfile.gettempdir(), "dreamlab_b200_bench_models"))
    name = "sd15-lcm" if c["arch"] == "sd15" else "sdxl-base"
    path = os.path.join(root, name)
    done = os.path.join(path, ".complete")
    if rank == 0 and not os.path.exists(done):
        if c["arch"] == "sd15":
            syn.write_model_dir(path)
            syn.write_text_encoder(path)        # CLIP ViT-L/14 text tower (random init): prompts go through it on the device
        else:
            syn.write_model_dir(path, syn.sdxl_unet_cfg(), syn.sdxl_vae_cfg())
        open(done, "w").close()
    barrier()
    return root, name


def make_pool(c, root, name, num_workers, device_env=None):
    import contextlib
    from backends.worker_factory import create_cuda_worker
    from backends.worker_pool import WorkerPool
    os.environ["MODEL_ROOT"], os.environ["MODEL"] = root, name
    if device_env:
        os.environ["CUDA_DEVICE"] = device_env
    else:
        os.environ.pop("CUDA_DEVICE", None)
    with contextlib.redirect_stdout(sys.stderr):          # the workers announce themselves with print()
        return WorkerPool(queue_max=1 << 16, worker_factory=create_cuda_worker, mode_config=_Modes(root, name),
                          registry=_Registry(), num_workers=num_workers, max_batch=c["batch"])


def pool_requests(pool, c, n, seed0):
    from backends.worker_pool import GenerationJob
    size = f"{c['size']}x{c['size']}"
    return [pool.submit_job(GenerationJob(req=SimpleNamespace(
        prompt=f"bench prompt {seed0 + i}", size=size, num_inference_steps=c["lcm_steps"],
        guidance_scale=c["gs"], seed=seed0 + i))) for i in range(n)]


def pool_e2e(pool, c, n_requests, warm_requests, before_timed=None):
    """-> (seconds for n_requests, mean PNG bytes).  Requests in (host objects), PNG bytes out."""
    for f in pool_requests(pool, c, warm_requests, 0):          # graph capture, encoder threads, allocator
        f.result(timeout=1200)
    if before_timed is not None:
        before_timed()
    t0 = time.perf_counter()
    outs = [f.result(timeout=1200) for f in pool_requests(pool, c, n_requests, 100000)]
    dt = time.perf_counter() - t0
    for png, _seed in outs[:2]:
        assert png[:8] == b"\x89PNG\r\n\x1a\n"
    return dt, sum(len(o[0]) for o in outs) / len(outs)


# ------------------------------------------------------------------------------------------------
# B200 arm, SD1.5 configs (C2 / C3 / C4 shard)
# ------------------------------------------------------------------------------------------------
def run_b200(args, c):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    from dreamlab_b200 import lib as _lib
    _lib.wait_for_driver()
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device; the b200 arm has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    _lib.load()         # the library __graft_entry__.build() compiled: nothing is compiled at run time
    if c["arch"] == "sdxl":
        return run_b200_c5(args, c, rank, local, world, dev, barrier, max_over_ranks)
    from dreamlab_b200 import lib
    from dreamlab_b200.engine import LCMPipelineB200
    from dreamlab_b200 import synthetic as syn
    from dreamlab_b200.synthetic import synthetic_inputs
    B, size, nsteps = c["batch"], c["size"], c["lcm_steps"]
    GFLOP_IMAGE = gflop_image(c)
    ucfg, vcfg = syn.sd15_lcm_unet_cfg(), syn.sd_vae_cfg()
    pipe = LCMPipelineB200(syn.random_state_dict(syn.unet_shapes(ucfg), 0), ucfg,
                           syn.random_state_dict(syn.vae_decoder_shapes(vcfg), 1), vcfg, dev)
    pe, lat, noise = synthetic_inputs(B, size, size, nsteps, seed_base=1000 + rank * B)
    gr = pipe.graph_for(B, size // 8, size // 8, nsteps)
    # ---- device-resident inputs (value) ----
    gr.pe.copy_(pe)
    gr.lat.copy_(lat)
    gr.noise.copy_(noise)
    from dreamlab_b200.scheduler import guidance_scale_embedding
    gr.w_emb.copy_(guidance_scale_embedding(torch.zeros(B), 256))
    l2_flush = torch.empty(256 * 1024 * 1024, device=dev, dtype=torch.uint8)   # > 126 MB L2

    for _ in range(max(args.warmup, 3)):
        gr.graph.replay()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
           for _ in range(args.steps)]
    barrier()
    for a, b in evs:
        l2_flush.zero_()                      # flush L2 between timed iterations
        a.record()
        gr.graph.replay()
        b.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # what generate(..., return_latents=True) hands its caller: u8 images NHWC and the final latents NHWC
        dump_outputs(args.dump_outputs, image=gr.img, latents=gr.final)
    step_ms = [a.elapsed_time(b) for a, b in evs]
    total_ms = max_over_ranks(sum(step_ms))
    value = world * B * args.steps / (total_ms / 1e3)

    # ---- e2e_engine: host pinned inputs -> engine API -> host image, every step ----
    pe_h, lat_h, noise_h = pe.pin_memory(), lat.pin_memory(), noise.pin_memory()
    img_h = torch.empty(B, size, size, 3, dtype=torch.uint8).pin_memory()
    h2d_engine = pe_h.numel() * 4 + lat_h.numel() * 4 + noise_h.numel() * 4 + B * 256 * 4

    def e2e_once():
        img = pipe.generate(pe_h, lat_h, noise_h, nsteps, 1.0, use_graph=True)
        img_h.copy_(img, non_blocking=True)
    for _ in range(2):
        e2e_once()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        e2e_once()
    e1.record()
    barrier()
    e2e_engine = world * B * args.steps / (max_over_ranks(e0.elapsed_time(e1)) / 1e3)

    # ---- roofline of the dominant kernel (igemm), CUDA events around every launch ----
    roof = None
    if rank == 0:
        lib.profile_begin()
        pipe.generate(gr.pe, gr.lat, gr.noise, nsteps, 1.0, use_graph=False)
        prof = lib.profile_end()
        sustained, burst, hbm, src = peaks()
        ig = prof.get("igemm", {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "n": 0})
        tot_ms = sum(v["ms"] for v in prof.values())
        ach = ig["flops"] / (ig["ms"] / 1e3) / 1e12 if ig["ms"] > 0 else 0.0
        # DRAM bytes per igemm launch from the committed ncu capture of this very workload; only quoted
        # for the configuration (and launch count) it was taken on
        traffic, traffic_src = None, None
        for tj_name in ("r02_ncu_dram_per_kernel.json", "r01_ncu_dram_per_kernel_v7.json"):
            tj = os.path.join(ROOT, "profiles", tj_name)
            if os.path.exists(tj) and (B, size, nsteps) == (16, 512, 4):
                k = json.load(open(tj)).get("dl::igemm_kernel")
                if k and k["launches"] == ig["n"]:
                    traffic = (k["dram_read_bytes"] + k["dram_write_bytes"]) / k["launches"]
                    traffic_src = f"profiles/{tj_name} (ncu, same workload, per launch)"
                    break
        roof = {"bound": "tensor", "kernel": "igemm_kernel (tcgen05 implicit-GEMM conv/linear)",
                "achieved": ach, "peak": sustained, "peak_kind": f"bf16 dense sustained, {src}",
                "unit": "TFLOP/s", "frac": ach / sustained, "traffic": traffic, "traffic_unit": "bytes/launch (DRAM)",
                "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": ig["bytes"] / ig["n"] if ig["n"] else None,
                "launches": ig["n"], "share_of_step": ig["ms"] / tot_ms if tot_ms else None,
                "step_achieved_tflops": GFLOP_IMAGE * value / world / 1e3,
                "step_frac": GFLOP_IMAGE * value / world / 1e3 / sustained,
                "by_kernel_ms": {k: round(v["ms"], 3) for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}}
        at = prof.get("attention")
        if at and at["ms"] > 0:
            tf = at["flops"] / (at["ms"] / 1e3) / 1e12
            roof["attention_kernel"] = {"bound": "tensor", "achieved": tf, "peak": sustained, "unit": "TFLOP/s",
                                        "frac": tf / sustained, "launches": at["n"], "ms": round(at["ms"], 3)}
        # the dominant HBM-bound kernel: one-pass GroupNorm(+SiLU) apply
        # (algorithmic 4 B/element: bf16 read once + written once), against the measured copy rate
        ga = prof.get("groupnorm_apply")
        if ga and ga["ms"] > 0:
            gbs = ga["bytes"] / (ga["ms"] / 1e3) / 1e9
            roof["hbm_kernel"] = {"bound": "hbm", "kernel": "gn_apply_kernel (GroupNorm+SiLU, one pass)",
                                  "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm,
                                  "launches": ga["n"], "ms": round(ga["ms"], 3)}

    # ---- single-request latency (B = 1, one CUDA-graph replay), p50 over 30 replays ----
    lat_b1 = None
    if rank == 0:
        pe1, l1, n1 = syn.synthetic_inputs(1, size, size, nsteps)
        run1 = lambda: pipe.generate(pe1, l1, n1, nsteps, 1.0, use_graph=True)   # noqa: E731
        for _ in range(3):
            run1()
        torch.cuda.synchronize()
        ts = []
        for _ in range(30):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            run1()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        lat_b1 = statistics.median(ts)
    launches_per_step = gr.launches
    del pipe, gr, l2_flush
    import gc
    gc.collect()
    torch.cuda.empty_cache()

    # ---- e2e through the plugin boundary: requests -> WorkerPool -> B200Worker -> PNG bytes ----
    e2e = None
    if not args.no_pool_e2e:
        root, name = bench_model_dir(c, rank, barrier)
        pool = make_pool(c, root, name, 1, device_env=f"cuda:{local}")
        n_req = B * args.steps
        # headline: the serving configuration for this box, PNG files assembled on the device (B200_PNG=gpu; an
        # explicit B200_PNG in the environment wins).  The reference's exact host call (PIL / zlib on encoder
        # threads) is measured right after on the same pool as `e2e_png_pil`
        png_mode = os.environ.get("B200_PNG", "").strip().lower() or "gpu"
        os.environ["B200_PNG"] = png_mode
        barrier()
        dt, png_bytes = pool_e2e(pool, c, n_req, 2 * B)
        barrier()
        dt = max_over_ranks(dt)
        e2e_pil = None
        if png_mode != "pil":
            os.environ["B200_PNG"] = "pil"
            n_pil = B * min(args.steps, 6)
            barrier()
            dt_p, bytes_p = pool_e2e(pool, c, n_pil, B)
            barrier()
            e2e_pil = {"value": world * n_pil / max_over_ranks(dt_p), "unit": UNIT, "png": "pil", "png_bytes_mean": bytes_p,
                       "requests": n_pil * world,
                       "note": "same pool, the reference's img.save(buf, format='PNG') on the host encoder threads"}
            os.environ["B200_PNG"] = png_mode
        pool.shutdown()
        e2e = {"value": world * n_req / dt, "unit": UNIT,
               # per step (= one batch of B requests) over all ranks, like `value`: what enters from the host is the
               # request itself — 77 int64 token ids per prompt (hashed stand-in ids: no vocabulary offline) and the
               # seed; the CLIP text tower runs on the device, latents / step noise are drawn on the device from the
               # request's seed exactly as the reference's CUDA worker does (`cuda_worker.py:212-213`); what leaves is
               # the PNG file (device-side writer) or the u8 image (PIL encoder threads)
               "h2d_bytes_per_step": world * (B * 77 * 8 + B * 8),
               "d2h_bytes_per_step": world * B * size * size * 3,
               "path": "GenerationJob(prompt, seed) -> WorkerPool.submit_job -> B200Worker.run_batch (token ids -> CLIP-L "
                       "text tower on the device -> LCM loop -> VAE) -> PNG bytes",
               "png": png_mode, "png_bytes_mean": png_bytes,
               "requests": n_req * world, "timed": "wall clock, first submit to last PNG, max over ranks",
               "host_cores": os.cpu_count()}
        if e2e_pil is not None:
            e2e["e2e_png_pil"] = e2e_pil

    # ---- CPU baseline (rank 0, N=1 only): 1 warm-up + median of 3 full oracle passes ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        once, txt, extrapolated = cpu_reference(c, threads)
        once()
        runs = [once() for _ in range(3)]
        per_image = statistics.median(r[1] for r in runs)
        cpu = {"value": 1.0 / per_image, "unit": UNIT, "cores": threads, "kind": "port", "sample": txt,
               "seconds_per_image_runs": [round(r[1], 3) for r in runs], "extrapolated": extrapolated}

    if rank == 0:
        print(json.dumps({
            "metric": c["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": workload_text(c),
                       "batch_per_gpu": B, "global_batch": B * world, "l2": "flushed between timed iterations",
                       "cuda_graph": True, "parallelism": f"replicas x{world} (no collective)"},
            "p50_latency_ms_per_batch": statistics.median(step_ms),
            "p50_latency_ms_single_image": lat_b1,
            "e2e": e2e if e2e is not None else {"value": e2e_engine, "unit": UNIT, "h2d_bytes_per_step": world * h2d_engine,
                                                "d2h_bytes_per_step": world * img_h.numel(),
                                                "path": "engine (pool e2e skipped)"},
            "e2e_engine": {"value": e2e_engine, "unit": UNIT, "h2d_bytes_per_step": world * h2d_engine,
                           "d2h_bytes_per_step": world * img_h.numel(),
                           "path": "pinned host tensors -> LCMPipelineB200.generate (CUDA graph) -> pinned host u8"},
            "gpu_launches": launches_per_step * args.steps * world,
            "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
        }))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# B200 arm, config C5: one SDXL 1024^2 image over the ranks
# ------------------------------------------------------------------------------------------------
def run_b200_c5(args, c, rank, local, world, dev, barrier, max_over_ranks):
    import torch
    from dreamlab_b200 import lib
    from dreamlab_b200 import patch_parallel as pp
    from dreamlab_b200 import synthetic as syn
    from dreamlab_b200.engine import LCMPipelineB200
    size, nsteps, gs = c["size"], c["lcm_steps"], c["gs"]
    ucfg, vcfg = syn.sdxl_unet_cfg(), syn.sdxl_vae_cfg()
    pipe = LCMPipelineB200(syn.random_state_dict(syn.unet_shapes(ucfg), 0, torch.bfloat16), ucfg,
                           syn.random_state_dict(syn.vae_decoder_shapes(vcfg), 1, torch.bfloat16), vcfg, dev)
    pdim = ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim
    pe, lat, noise = syn.synthetic_inputs(1, size, size, nsteps, ctx_dim=ucfg.cross_attention_dim)
    pooled = torch.randn(1, pdim, generator=torch.Generator().manual_seed(2))
    pe_h, lat_h, noise_h, pooled_h = (t.pin_memory() for t in (pe, lat, noise, pooled))
    pe_d, lat_d, noise_d, pooled_d = (t.to(dev) for t in (pe, lat, noise, pooled))
    img_h = torch.empty(1, size, size, 3, dtype=torch.uint8).pin_memory()
    peer = os.environ.get("B200_C5_EXCHANGE", "peer") == "peer"
    group = args.c5_group if args.c5_group and args.c5_group < world else world
    n_groups = world // group
    if world > 1 and group != world:
        # throughput layout: the ranks form n_groups independent groups, each sharding ITS OWN image (group = 2:
        # the two CFG halves of one image per GPU pair, one noise-prediction exchange per step, no strips)
        import torch.distributed as dist
        if group != 2 or world % 2:
            raise RuntimeError("--c5-group supports groups of 2 ranks (the CFG pair)")
        groups = [dist.new_group(list(range(i * group, (i + 1) * group))) for i in range(n_groups)]
        mine = groups[rank // group]
        den = pp.PatchParallelDenoiser(pipe, pp.PeerComm(mine) if peer else pp.DistComm(mine))
    elif world > 1:
        den = pp.dist_denoiser(pipe, peer=peer)
    if world > 1:
        def step(host: bool):
            a = (pe_h, pooled_h, lat_h, noise_h) if host else (pe_d, pooled_d, lat_d, noise_d)
            img = den.generate(*a, nsteps, gs, use_graph=True, vae_strips=True)
            if host:
                img_h.copy_(img, non_blocking=True)
            return img
    else:
        def step(host: bool):
            a = (pe_h, lat_h, noise_h) if host else (pe_d, lat_d, noise_d)
            img = pipe.generate(*a, nsteps, gs, use_graph=True, pooled_embeds=pooled_h if host else pooled_d)
            if host:
                img_h.copy_(img, non_blocking=True)
            return img
    n0 = lib.launch_count
    for _ in range(max(args.warmup, 3)):
        step(False)
    barrier()
    launches = None
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l2_flush = torch.empty(256 * 1024 * 1024, device=dev, dtype=torch.uint8)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for a, b in evs:
        l2_flush.zero_()
        a.record()
        img = step(False)
        b.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, image=img)
    step_ms = [a.elapsed_time(b) for a, b in evs]
    total_ms = max_over_ranks(sum(step_ms))
    value = n_groups * args.steps / (total_ms / 1e3)
    for _ in range(2):
        step(True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step(True)
    e1.record()
    barrier()
    e2e_v = n_groups * args.steps / (max_over_ranks(e0.elapsed_time(e1)) / 1e3)
    # launches of one eager pass on this rank (the graph replays exactly these)
    n0 = lib.launch_count
    if world > 1:
        den.generate(pe_d, pooled_d, lat_d, noise_d, nsteps, gs, use_graph=False, vae_strips=True)
    else:
        pipe.generate(pe_d, lat_d, noise_d, nsteps, gs, pooled_embeds=pooled_d)
    barrier()
    launches = lib.launch_count - n0
    if rank == 0:
        sustained, burst, hbm, src = peaks()
        tf = gflop_image(c) * value / 1e3
        print(json.dumps({
            "metric": c["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if n_groups == 1 else "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload_text(c), "l2": "flushed between timed iterations", "cuda_graph": True,
                       "images_in_flight": n_groups,
                       "parallelism": ("1 GPU" if world == 1 else
                                       f"{n_groups} independent groups of {group} ranks, one image each (CFG halves on the "
                                       f"two GPUs of a pair, one exchange per step)" if n_groups > 1 else
                                       f"CFG halves x row strips over {world} ranks, exchanges: "
                                       f"{'NVLink peer-memory kernels' if peer else 'ncclAllGather'}; VAE decode as row strips")},
            "ms_per_unet_step": total_ms / args.steps / nsteps,
            "e2e": {"value": e2e_v, "unit": UNIT,
                    "h2d_bytes_per_step": 4 * (pe.numel() + lat.numel() + noise.numel() + pooled.numel()),
                    "d2h_bytes_per_step": img_h.numel(),
                    "path": "pinned host tensors -> PatchParallelDenoiser.generate (CUDA graph) -> pinned host u8"},
            "gpu_launches": launches * args.steps * world,
            "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "whole pass (igemm + attention dominate)", "achieved": tf / world,
                         "peak": sustained, "unit": "TFLOP/s per GPU", "frac": tf / world / sustained,
                         "peak_kind": f"bf16 dense sustained, {src}", "traffic": None},
            "cpu_baseline": None,
        }))
    sys.stdout.flush()
    os._exit(0)        # NCCL collectives captured in CUDA graphs: communicator teardown can hang


# ------------------------------------------------------------------------------------------------
# ONE process, N GPU workers behind one WorkerPool (the product's multi-GPU path)
# ------------------------------------------------------------------------------------------------
def run_pool(args, c):
    import torch
    from dreamlab_b200 import lib as _lib
    _lib.wait_for_driver()
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device; the b200 arm has no CPU fallback")
    _lib.load()
    n = args.pool_workers
    ngpu = min(n, torch.cuda.device_count())      # more workers than GPUs: worker k runs on cuda:(k % GPUs)
    os.environ["B200_PNG"] = os.environ.get("B200_PNG", "").strip().lower() or "gpu"
    root, name = bench_model_dir(c, 0, lambda: None)
    pool = make_pool(c, root, name, n)
    B = c["batch"]
    n_req = n * B * args.steps
    # clocks / throttle reasons of EVERY GPU during the timed region: eight GPUs running back to back in one box
    # is also a box-level power question
    samplers = [ClockSampler(i) for i in range(ngpu)]
    dt, png_bytes = pool_e2e(pool, c, n_req, 2 * n * B, before_timed=lambda: [sp.start() for sp in samplers])
    clocks = [sp.stop() for sp in samplers]
    pool.shutdown()
    v = n_req / dt
    if os.environ.get("B200_BATCH_TIMING", "0") not in ("0", "", "false"):
        from backends.b200_worker import batch_timing_summary
        print(json.dumps({"batch_timing": batch_timing_summary()}), file=sys.stderr)
    print(json.dumps({
        "metric": c["metric"], "value": v, "unit": UNIT, "n_gpus": ngpu, "steps": args.steps, "warmup": 2,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": workload_text(c), "parallelism": f"ONE process, WorkerPool with {n} B200Worker threads "
                   f"on {ngpu} GPU(s) (worker k on cuda:(k % GPUs)), shared FIFO, micro-batches of {B}, PNG on encoder threads / GPU",
                   "png": os.environ.get("B200_PNG", "pil"), "host_cores": os.cpu_count()},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": n * (B * 77 * 8 + B * 8),
                "d2h_bytes_per_step": n * B * c["size"] * c["size"] * 3, "png_bytes_mean": png_bytes,
                "path": "GenerationJob(prompt, seed) -> WorkerPool.submit_job -> B200Worker.run_batch (token ids -> "
                        "CLIP-L text tower on the device -> LCM loop -> VAE) -> PNG bytes",
                "requests": n_req, "timed": "wall clock, first submit to last PNG"},
        "gpu_launches": None,
        "clocks": {"per_gpu_sm_mhz": [k["sm_mhz"] for k in clocks], "sm_max_mhz": clocks[0]["sm_max_mhz"],
                   "reasons": sorted({r for k in clocks for r in k["reasons"]}),
                   "samples": [k.get("samples") for k in clocks]},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="override the config's batch per GPU")
    ap.add_argument("--size", type=int, default=0)
    ap.add_argument("--lcm-steps", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pool-e2e", action="store_true", help="skip the WorkerPool/PNG leg (kernel work only)")
    ap.add_argument("--c5-group", type=int, default=0,
                    help="config c5: ranks per image (default: all ranks shard ONE image); 2 = one image per GPU pair")
    ap.add_argument("--pool-workers", type=int, default=0,
                    help="one process, WorkerPool with this many GPU workers; prints the e2e line only")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32, "
                         f"at most {DUMP_BYTES_MAX // 10**6} MB in all; b200 arm, --config c2 / c3 / c5)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.pool_workers):
        ap.error("--dump-outputs: the b200 arm's timed path only (not --impl reference or --pool-workers)")
    c = dict(CONFIGS[args.config])
    if args.batch:
        c["batch"] = args.batch
    if args.size:
        c["size"] = args.size
    if args.lcm_steps:
        c["lcm_steps"] = args.lcm_steps
    if args.impl == "reference":
        run_reference(args, c)
    elif args.pool_workers:
        run_pool(args, c)
    else:
        run_b200(args, c)


if __name__ == "__main__":
    main()
