#!/usr/bin/env python
"""bench.py -- diffusion iter/s of the b200sd hot path on N B200s (one process per GPU).

A "step" is one denoising iteration of BASELINE.json configs[1] (SD-2.1-base txt2img, 512x512, 20 DDIM
steps, CFG 7.5, fp16): UNet forward at batch 2 (uncond, cond) + the fused CFG/scheduler-step kernel,
i.e. the reference's "Diffusion Speed (iter/s)" (README.md:65,83).  `value` is measured with all inputs
resident in HBM; `e2e` is the same iteration driven through the reference-facing model-call boundary
(`unet(sample=np, timestep=np, encoder_hidden_states=np)["noise_pred"]`, coreml_model.py:118-120) with
pinned HOST buffers, host<->device copies inside the timed region.  Extra keys report 512^2 images/s
(20 steps + VAE decode), the tensor-core roofline of the dominant kernel and the CPU baseline.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

--dump-outputs DIR writes, after the timed steps, what the timed paths computed in their last step as DIR/<name>.npy
(float32): `latents` and `noise_pred` (the UNet output, rows uncond / cond) of the device loop, `e2e_latents` and
`e2e_noise_pred` of the boundary loop, `image` (the last decoded image of the images/s loop); `noise_pred` alone
for `--impl reference`.  All inputs derive from fixed seeds, so two builds run with the same arguments can be
compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

UNET_TFLOP = 1.609          # SURVEY 8(d): algorithmic FLOPs of one SD-2.1-base UNet forward at B=2
VAE_TFLOP = 2.51
PUBLISHED_ITER_S = 3.07     # BASELINE.md section 1: best published SD-2.1-base 512^2 (iPad Pro M2, Core ML)
WORKLOAD = "SD-2.1-base txt2img 512x512, 20 DDIM steps, CFG 7.5, fp16 (BASELINE configs[1])"


def CONFIG(world):
    """The `config` object of the JSON line: identical for the b200sd arm and the reference arm."""
    return {"workload": WORKLOAD, "unet_batch": 2, "latent": "4x64x64", "text_tokens": 77,
            "weights": "random-init SD-2.1-base (865.9 M params)",
            "parallelism": f"replicas x{world}, independent prompts per rank, no data-path collective",
            "cache": "inputs larger than L2: every step streams 1.73 GB of fp16 weights through the 126 MB L2"}


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d["bf16_tflops"], d["bf16_tflops_sustained"], d["hbm_gbs"], "measured"
    return 1590.0, 1400.0, 6650.0, "fallback"


def dump_outputs(out_dir, arrays):
    """DIR/<name>.npy in float32 for every array (a few MB in all; the bound keeps dumps comparable and small)."""
    arrays = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in arrays.items()}
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active") and not v.lower().startswith("not"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own PyTorch-CPU UNet (or its restatement when the tree is absent)
# ------------------------------------------------------------------------------------------------
def cpu_unet_runner():
    from b200sd import config
    from oracle import ref_unet, restated

    cfg = config.SD21_BASE_UNET
    sd = config.random_state_dict(config.unet_param_shapes(cfg), seed=1)
    g = torch.Generator().manual_seed(2)
    x = torch.randn(2, 4, 64, 64, generator=g)
    c = torch.randn(2, 1024, 1, 77, generator=g)
    t = torch.tensor([981.0, 981.0])
    torch.set_grad_enabled(False)
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm should use the host's cores (physical ~ logical / 2)
    torch.set_num_threads(max(1, (os.cpu_count() or 2) // 2))
    if ref_unet.available():
        m = ref_unet.build_unet(cfg, sd, impl="ORIGINAL")
        return "reference", (lambda: m(x, t, c)[0])
    return "port", (lambda: restated.unet_forward(sd, cfg, x, t, c))


def time_cpu(budget_s=25.0, max_steps=3, warmup=1):
    kind, fn = cpu_unet_runner()
    for _ in range(warmup):
        fn()
    times = []
    t_start = time.perf_counter()
    while len(times) < max_steps and (not times or time.perf_counter() - t_start + times[-1] < budget_s):
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
    best = min(times)
    return {"value": round(1.0 / best, 4), "unit": "iter/s", "cores": torch.get_num_threads(), "kind": kind,
            "sample": f"{len(times)} timed fp32 UNet forwards (SD-2.1-base, bs=2, 64x64 latents, t=981; best of "
                      f"{len(times)}, median {sorted(times)[len(times) // 2]:.2f} s) after {warmup} warm-up",
            "cpu_count": os.cpu_count()}, times


def run_reference_arm(args, rank, world):
    """`--impl reference`: the reference's own CPU implementation of the path (its unmodified PyTorch-CPU UNet modules
    when $B200SD_REFERENCE names a reference checkout, else the oracle restatement of them) on the box's host cores,
    same `config`, metric and unit as the b200sd arm, EXACTLY --steps timed UNet forwards after --warmup untimed ones (a CPU
    forward takes seconds: the default 40 + 3 finish within a few minutes).  Rank 0 only."""
    if rank != 0:
        return
    kind, fn = cpu_unet_runner()
    warm = max(0, args.warmup)
    for _ in range(warm):
        fn()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = fn()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"noise_pred": out.numpy()})
    val = args.steps / dt
    line = {
        "impl": "reference", "metric": "diffusion_iter_per_s", "value": round(val, 4), "unit": "iter/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": warm, "ms_per_step": round(1e3 * dt / args.steps, 2),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": round(val / PUBLISHED_ITER_S, 4),
        "dtype": "f32", "data": "synthetic",
        "config": CONFIG(max(1, args.gpus)),
        "cpu_baseline": {"value": round(val, 4), "unit": "iter/s", "cores": torch.get_num_threads(), "kind": kind,
                         "sample": f"{args.steps} fp32 UNet forwards (SD-2.1-base, bs=2, 64x64 latents) of the reference's "
                                   f"PyTorch-CPU path ({'unmodified reference modules' if kind == 'reference' else 'oracle restatement (port)'}); "
                                   "the CPU arm runs the UNet forward only (the reference does CFG + scheduler math on "
                                   "the host as well; negligible)"},
        "e2e": {"value": round(val, 4), "unit": "iter/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
N_STEPS_IMG, GUIDANCE = 20, 7.5


class LoopBench:
    """K denoising iterations of a pipeline's device loop as ONE CUDA graph.  Every 20 iterations (one image) the
    graph re-runs the per-prompt prologue (cross-attention K/V, time-embedding table, first UNet input), exactly
    what ``B200StableDiffusionPipeline.denoise`` captures; optional ControlNets run inside every step."""

    def __init__(self, pipe, lat0, cond=None):
        from b200sd import lib as L
        from b200sd import scheduler as S
        self.L, self.pipe, self.lat0 = L, pipe, lat0
        self.plan = S.DDIMScheduler(N_STEPS_IMG).plan()
        self.cond = cond
        self.graphs = {}

    def body(self, k_steps, first=0):
        L, pipe = self.L, self.pipe
        u, n = pipe.unet, pipe.images_per_call
        table = getattr(self, "_table", None)
        for i in range(first, first + k_steps):
            j = i % N_STEPS_IMG
            if j == 0:
                pipe._latents.copy_(self.lat0)
                pipe._hist.zero_()
                u.prepare_prompt()
                table = self._table = u.time_table(self.ts_rows)
                L.nchw_to_nhwc(pipe._latents, c_pad=u.engine.in_pad, out=u._x_nhwc[:n])
                L.nchw_to_nhwc(pipe._latents, c_pad=u.engine.in_pad, out=u._x_nhwc[n:])
                if self.cond is not None:
                    pipe.prepare_controlnets(self.ts_rows)
            st = self.plan[j]
            res = pipe.controlnet_residuals(j, table[j]) if self.cond is not None else None
            u._run_core(table[j], res)
            k = pipe._coeffs(st, GUIDANCE)
            k.noise_pred_nhwc = 1
            k.n_hist, k.push_eps_slot, k.push_x0_slot, k.push_x_slot = 0, -1, -1, -1
            L.cfg_scheduler_step(u._out_nhwc, pipe._latents, k, unet_in=u._x_nhwc)

    def profile_one_step(self):
        """For ``ncu --profile-from-start off``: warm up eagerly, then run exactly ONE mid-image iteration (the launch
        sequence every timed step replays; no per-prompt prologue) between cudaProfilerStart / Stop."""
        self.ts_rows = self.pipe._ts_rows(self.plan)
        if self.cond is not None:
            self.pipe.set_control_conditions(self.cond)
        self.body(2)
        torch.cuda.synchronize()
        n0 = self.L.launch_count()
        torch.cuda.profiler.start()
        self.body(1, first=2)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return self.L.launch_count() - n0

    def capture(self, k_steps, classes=0xF):
        key = (k_steps, classes)
        if key in self.graphs:
            return self.graphs[key]
        L, pipe = self.L, self.pipe
        self.ts_rows = pipe._ts_rows(self.plan)
        if self.cond is not None:
            pipe.set_control_conditions(self.cond)
        s = torch.cuda.Stream(device=pipe.device)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            n0 = L.launch_count()
            self.body(min(k_steps, 2))   # eager warm-up: workspaces, weight tiling, kernel attributes
            torch.cuda.synchronize()
            n1 = L.launch_count()
            self.body(N_STEPS_IMG)       # launch census of one whole image
            self.launches_per_image = L.launch_count() - n1
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        L.load().b200sd_set_launch_classes(classes)
        try:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.body(k_steps)
        finally:
            L.load().b200sd_set_launch_classes(0xF)
        self.graphs[key] = g
        return g


def timed_replays(graph, reps, barrier):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(2):
        graph.replay()
    barrier()
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record()
    barrier()
    return e0.elapsed_time(e1) / reps


def gemm_census(pipe):
    """Algorithmic FLOPs (2 M N K) of every tensor-core GEMM / convolution launch of one UNet forward."""
    from b200sd import lib as L
    recs = []
    orig = L.run_gemm

    def rec(args):
        m = args.m if (args.mode == 0 and not args.halo) else args.n_img * (args.h // max(1, args.stride)) * (args.w // max(1, args.stride))
        k = (args.c0 + args.c1) * (9 if args.mode == 1 else 1) + args.c2 + args.c3  # (+ a folded shortcut)
        recs.append(2.0 * m * args.n * k)
        orig(args)

    L.run_gemm = rec
    try:
        u = pipe.unet
        u._run_core(torch.zeros(u.batch, u.engine.temb_total, device=pipe.device))
    finally:
        L.run_gemm = orig
    torch.cuda.synchronize()
    return sum(recs), len(recs)


def class_breakdown(loop, barrier, peaks, pipe):
    """Device time of one image's loop (20 steps + prologue) with only ONE kernel class launching, per class: the
    same launch sequence on the same buffers, each class captured as its own CUDA graph.  No event gaps, no profiler
    serialisation: the four numbers add up to the full loop when the classes do not overlap."""
    out = {}
    for name, bit in (("gemm_conv", 1), ("attention", 2), ("normalisation", 4), ("elementwise", 8)):
        g = loop.capture(N_STEPS_IMG, classes=bit)
        out[name] = round(timed_replays(g, 3, barrier) / N_STEPS_IMG, 4)
    flops, launches = gemm_census(pipe)
    burst, sustained, _, how = peaks
    ms = out["gemm_conv"]
    achieved = flops / (ms * 1e-3) / 1e12
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic_r2.json")) as f:
            traffic = round(json.load(f)["dram_bytes_per_launch"])
    except (OSError, KeyError, ValueError):
        pass
    roof = {"bound": "tensor", "kernel": "umma_gemm_kernel + halo_conv_kernel (every conv3x3 / 1x1 / linear launch of one UNet forward)",
            "achieved": round(achieved, 1), "peak": sustained, "unit": "TFLOP/s", "frac": round(achieved / sustained, 4),
            "peak_kind": f"{how} sustained bf16 dense (kernels timed inside a long step)", "traffic": traffic,
            "traffic_unit": "DRAM bytes per launch (ncu; algorithmic = weights 1.73e9 B / forward)",
            "launches": launches, "algorithmic_tflop": round(flops / 1e12, 4), "kernel_ms_sum": ms,
            "how": "CUDA-graph replay of the loop with only the GEMM / convolution class launching (same buffers, no "
                   "event gaps), divided by the steps"}
    return out, roof


def extra_config(name, dev, barrier, peaks, steps=N_STEPS_IMG):
    """BASELINE configs[3] (SDXL-base 768x768) and configs[4] (SD-2.1 + ControlNet): iter/s of the device loop."""
    from b200sd import config as C
    from b200sd.pipeline import B200StableDiffusionPipeline
    g = torch.Generator().manual_seed(7)
    if name == "sdxl_768":
        pipe = B200StableDiffusionPipeline.from_random_init("sdxl-base", images_per_call=1, device=dev, seed=1,
                                                            scheduler="DDIM", height=768, width=768)
        tflop, hw, d_ctx, cond = 7.282, 96, 2048, None
        pipe.unet._time_ids.copy_(torch.tensor([[768, 768, 0, 0, 768, 768]] * 2, dtype=torch.float32))
        pipe.unet._text_embeds.copy_(torch.randn(2, 1280, generator=g))
    else:
        pipe = B200StableDiffusionPipeline.from_random_init("sd21-base", images_per_call=1, device=dev, seed=1,
                                                            scheduler="DDIM", controlnet_cfgs=[C.SD21_CONTROLNET])
        tflop, hw, d_ctx = 1.609 + 0.567, 64, 1024
        cond = [torch.rand(2, 3, 512, 512, generator=g).half().to(dev)]
    pipe.unet._ctx.copy_(torch.cat([torch.zeros(1, d_ctx, 1, 77), torch.randn(1, d_ctx, 1, 77, generator=g)]).half())
    lat0 = torch.randn(1, 4, hw, hw, generator=g).half().float().to(dev)
    loop = LoopBench(pipe, lat0, cond)
    ms = timed_replays(loop.capture(steps), 2, barrier) / steps
    _, sustained, _, _ = peaks
    return {"iter_per_s": round(1e3 / ms, 2), "ms_per_step": round(ms, 4),
            "launches_per_step": round(loop.launches_per_image / N_STEPS_IMG, 1),
            "step_roofline": {"algorithmic_tflop": tflop, "achieved": round(tflop / (ms * 1e-3), 1), "peak": sustained,
                              "unit": "TFLOP/s", "frac": round(tflop / (ms * 1e-3) / sustained, 4)}}


def run_gpu_arm(args, rank, local_rank, world):
    import torch.distributed as dist
    from b200sd import lib as L
    from b200sd.pipeline import B200StableDiffusionPipeline

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L.load()
    peaks = _peaks()
    pipe = B200StableDiffusionPipeline.from_random_init("sd21-base", images_per_call=1, device=dev, seed=1,
                                                        scheduler="DDIM")
    unet = pipe.unet
    g = torch.Generator().manual_seed(93 + rank)  # each rank = an independent prompt / seed (SURVEY 8e)
    emb_cond = torch.randn(1, 1024, 1, 77, generator=g)
    emb = torch.cat([torch.zeros_like(emb_cond), emb_cond]).half()
    lat0 = torch.randn(1, 4, 64, 64, generator=g).half().float().to(dev)
    unet._ctx.copy_(emb)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: K iterations of the pipeline's device loop (UNet forward bs=2 + fused CFG/DDIM step), one graph ----
    loop = LoopBench(pipe, lat0)
    if args.profile_step:
        print(json.dumps({"profile_step": True, "launches": loop.profile_one_step()}), flush=True)
        return
    graph = loop.capture(args.steps)
    launches_per_step = loop.launches_per_image / N_STEPS_IMG
    for _ in range(max(1, (max(3, args.warmup) + args.steps - 1) // args.steps)):  # >= W warm-up steps
        graph.replay()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    graph.replay()                      # EXACTLY args.steps iterations
    e1.record()
    barrier()
    ms_dev = e0.elapsed_time(e1)
    outputs = {}
    if args.dump_outputs and rank == 0:
        outputs["latents"] = pipe._latents.cpu().numpy()
        outputs["noise_pred"] = unet._out_nhwc.permute(0, 3, 1, 2).cpu().numpy()
    if args.quick:
        if rank == 0:
            if args.dump_outputs:
                dump_outputs(args.dump_outputs, outputs)
            print(json.dumps({"quick": True, "iter_per_s": round(world * args.steps / (ms_dev * 1e-3), 2),
                              "ms_per_step": round(ms_dev / args.steps, 4), "launches_per_step": round(launches_per_step, 1),
                              "fused": os.environ.get("B200SD_FUSED", "ln"), "pdl": os.environ.get("B200SD_PDL", "1")}),
                  flush=True)
        sampler.stop()
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- e2e: the reference-facing boundary call with pinned host buffers, copies inside the timed region ----
    from b200sd import scheduler as S
    plan = S.DDIMScheduler(N_STEPS_IMG).plan()
    h_sample = torch.empty(2, 4, 64, 64, dtype=torch.float16).pin_memory()
    h_t = torch.empty(2, dtype=torch.float16).pin_memory()
    h_ctx = emb.clone().pin_memory()
    h_lat = lat0.cpu().clone()
    np_sample, np_t, np_ctx = h_sample.numpy(), h_t.numpy(), h_ctx.numpy()

    def e2e_step(i):
        st = plan[i % N_STEPS_IMG]
        np_sample[:] = np.concatenate([h_lat.numpy()] * 2).astype(np.float16)
        np_t[:] = float(st.timestep)
        out = unet(sample=np_sample, timestep=np_t, encoder_hidden_states=np_ctx)["noise_pred"]  # H2D + D2H inside
        eps = out[:1] + GUIDANCE * (out[1:] - out[:1])          # host CFG + DDIM exactly like pipeline.py:559-569
        lat = st.cx * h_lat.numpy() + st.ce * eps
        h_lat.copy_(torch.from_numpy(lat))
        if (i + 1) % N_STEPS_IMG == 0:
            h_lat.copy_(lat0.cpu())
        return out, lat

    for i in range(3):
        e2e_step(i)
    barrier()
    t0 = time.perf_counter()
    e0.record()
    for i in range(args.steps):
        last = e2e_step(i)
    e1.record()
    barrier()
    ms_e2e = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
    if outputs:
        outputs["e2e_noise_pred"], outputs["e2e_latents"] = last
    clocks = sampler.stop()

    # ---- images/s: 20 steps + VAE decode through the public device-resident pipeline loop, >= 5 images ----
    def one_image():
        final = pipe.denoise(emb, lat0, N_STEPS_IMG, GUIDANCE)
        return pipe.decode_latents(final)

    one_image()
    barrier()
    n_img = 5
    e0.record()
    for _ in range(n_img):
        img = one_image()
    host_img = img.cpu()
    e1.record()
    barrier()
    ms_img = e0.elapsed_time(e1) / n_img
    if outputs:
        outputs["image"] = host_img.numpy()

    # ---- BASELINE configs[2] shape: 8 prompts per GPU (UNet batch 16), 20 steps + VAE decode of all 8 ----
    ms_b8 = float("nan")
    if not args.no_batched:
        pipe8 = B200StableDiffusionPipeline.from_random_init("sd21-base", images_per_call=8, device=dev, seed=1,
                                                             scheduler="DDIM")
        emb8 = torch.cat([torch.zeros(8, 1024, 1, 77), torch.randn(8, 1024, 1, 77, generator=g)]).half()
        lat8 = torch.randn(8, 4, 64, 64, generator=g).half().float()

        def eight_images():
            return pipe8.decode_latents(pipe8.denoise(emb8, lat8, N_STEPS_IMG, GUIDANCE))

        eight_images()
        barrier()
        e0.record()
        for _ in range(2):
            img8 = eight_images()
        img8_host = img8.cpu()
        e1.record()
        barrier()
        ms_b8 = e0.elapsed_time(e1) / 2
        del pipe8, eight_images, img8, img8_host
        torch.cuda.empty_cache()

    # max over ranks
    stats = torch.tensor([ms_dev, ms_e2e, ms_img, ms_b8], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e, ms_img, ms_b8 = [float(v) for v in stats.tolist()]

    # ---- rank 0 at N = 1: per-class attribution, the other BASELINE configs, the CPU arm ----
    classes = roof = None
    extra = {}
    if rank == 0:
        classes, roof = class_breakdown(loop, torch.cuda.synchronize, peaks, pipe)
    if world == 1 and not args.no_extra:
        del loop, graph
        torch.cuda.empty_cache()
        for name in ("sd21_controlnet", "sdxl_768"):
            try:
                extra[name] = extra_config(name, dev, torch.cuda.synchronize, peaks)
            except Exception as exc:  # reported, never hidden
                extra[name] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
            torch.cuda.empty_cache()

    if rank == 0:
        cpu, _ = time_cpu() if world == 1 else (None, None)
        value = world * args.steps / (ms_dev * 1e-3)
        e2e_val = world * args.steps / (ms_e2e * 1e-3)
        burst, sustained, hbm, how = peaks
        line = {
            "metric": "diffusion_iter_per_s", "value": round(value, 2), "unit": "iter/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": round(ms_dev / args.steps, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": round(value / PUBLISHED_ITER_S, 2),
            "dtype": "f16", "data": "synthetic",
            "config": CONFIG(world),
            "e2e": {"value": round(e2e_val, 2), "unit": "iter/s", "h2d_bytes_per_step": int(np_sample.nbytes +
                    np_t.nbytes + np_ctx.nbytes), "d2h_bytes_per_step": int(2 * 4 * 64 * 64 * 4),
                    "ms_per_step": round(ms_e2e / args.steps, 4), "api": "UNetModel.__call__(**np.ndarray) boundary + "
                    "host CFG/DDIM, as in the reference loop (pipeline.py:499-573)"},
            "gpu_launches": int(round(launches_per_step * args.steps)),
            "launches_per_step": round(launches_per_step, 1),
            "images_per_s": round(world * 1e3 / ms_img, 3),
            "ms_per_image": round(ms_img, 2),
            "images_timed": n_img,
            "batched_images_per_s": None if ms_b8 != ms_b8 else round(world * 8 * 1e3 / ms_b8, 3),
            "batched_note": "BASELINE configs[2] shape: 8 prompts per GPU (UNet batch 16), 20 DDIM steps + VAE decode",
            "step_roofline": {"bound": "tensor", "achieved": round(UNET_TFLOP / (ms_dev / args.steps * 1e-3), 1),
                              "peak": sustained, "unit": "TFLOP/s",
                              "frac": round(UNET_TFLOP / (ms_dev / args.steps * 1e-3) / sustained, 4),
                              "note": "whole UNet forward (1.609 TFLOP algorithmic) / device time per step; per GPU"},
            "roofline": roof,
            "kernel_class_ms_per_step": classes,
            "configs": extra or None,
            "cpu_baseline": cpu,
            "clocks": clocks,
            "image_checksum": float(host_img.double().sum()),
        }
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200sd", choices=["b200sd", "reference"])
    ap.add_argument("--no-batched", action="store_true", help="skip the 8-prompts-per-GPU images/s measurement")
    ap.add_argument("--quick", action="store_true", help="device-resident iter/s only (tuning runs; not a bench line)")
    ap.add_argument("--no-extra", action="store_true", help="skip the SDXL-768 / ControlNet configs (N = 1 only)")
    ap.add_argument("--profile-step", action="store_true",
                    help="run ONE eager denoising iteration between cudaProfilerStart/Stop (for ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's outputs as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__), *sys.argv[1:]]
        sys.exit(subprocess.call(cmd))
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: b200sd has no CPU fallback; use --impl reference for the CPU arm"}))
        sys.exit(1)
    run_gpu_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
