"""Sampler throughput on one GPU: loop-graph iter/s of every scheduler configuration, each timed right after DDIM so that
drift on a shared machine hits both alike, and the CUDA-event time of the step kernel with the sampler terms off, with
the input scale, and with the input scale + Philox noise (back-to-back launches inside one CUDA graph).  SD-2.1-base 512x512 (64x64 latents), random-init weights,
one image per call.  Prints one JSON document and writes it to --out.

    python tools/sampler_bench.py --steps 20 --rounds 3 --out out/sampler_bench.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from b200sd import lib as L  # noqa: E402
from b200sd import scheduler as S  # noqa: E402
from b200sd.pipeline import B200StableDiffusionPipeline  # noqa: E402

CONFIGS = [("DDIM", {}, 0.0), ("DDIM eta=1", {}, 1.0), ("DPMSolverMultistep", {"final_sigmas_type": "zero"}, 0.0),
           ("PNDM", {}, 0.0), ("EulerDiscrete", {}, 0.0), ("EulerAncestralDiscrete", {}, 0.0), ("LMSDiscrete", {}, 0.0)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def time_loop(pipe, name, kw, eta, emb, lat, steps, g, reps):
    pipe.scheduler_name, pipe.scheduler_kwargs = name.split(" ")[0], dict(kw)
    pipe.denoise(emb, lat, steps, g, eta=eta, seed=1)  # capture + warm-up
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for r in range(reps):
        pipe.denoise(emb, lat, steps, g, eta=eta, seed=1 + r)
    b.record()
    torch.cuda.synchronize()
    return steps * reps / (a.elapsed_time(b) / 1e3)


def time_kernel(variant, iters=2000):
    n, c, h, w = 1, 4, 64, 64
    eps = torch.randn(2 * n, h, w, c, device="cuda")
    lat = torch.randn(n, c, h, w, device="cuda")
    hist = torch.zeros(4, n, c, h, w, device="cuda")
    den = torch.empty_like(lat)
    ui = torch.zeros(2 * n, h, w, 8, dtype=torch.float16, device="cuda")
    key = torch.zeros(2, dtype=torch.int32, device="cuda")
    k = L.SamplerCoeffs()
    st = S.DDIMScheduler(20).plan()[5]
    k.step.guidance, k.step.cx, k.step.ce, k.step.x0_cx, k.step.x0_ce = 7.5, st.cx, st.ce, st.x0_cx, st.x0_ce
    k.step.push_eps_slot = k.step.push_x0_slot = k.step.push_x_slot = -1
    k.step.noise_pred_nhwc = 1
    k.in_scale = 1.0 if variant == "off" else 0.1
    k.noise_scale = 0.3 if variant == "noise" else 0.0
    for _ in range(50):
        L.sampler_step(eps, lat, k, hist=hist, denoised=den, unet_in=ui, rng_key=key)
    torch.cuda.synchronize()
    # launched from one CUDA graph, so the events time the device, not the host's per-call launch overhead
    per_graph = 200
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(per_graph):
            L.sampler_step(eps, lat, k, hist=hist, denoised=den, unet_in=ui, rng_key=key)
    g.replay()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters // per_graph):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / (iters // per_graph * per_graph)  # us per kernel


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sampler_bench needs a CUDA device")
    L.load()
    res = {"gpu": gpu_info(), "workload": f"sd21-base 512x512, 1 image, guidance 7.5, {args.steps} steps, loop graph",
           "kernel_us": {}, "iter_per_s": {}}
    for v in ("off", "scale", "noise"):
        res["kernel_us"][v] = round(time_kernel(v), 3)
    pipe = B200StableDiffusionPipeline.from_random_init("sd21-base", images_per_call=1, height=512, width=512, seed=0)
    emb = pipe._encode_prompt(["a photo of an astronaut riding a horse"], True, None)
    lat = np.random.RandomState(0).randn(1, 4, 64, 64).astype(np.float32)
    runs = {name: [] for name, _, _ in CONFIGS}
    ddim_pairs = {name: [] for name, _, _ in CONFIGS}
    for _ in range(args.rounds):
        for name, kw, eta in CONFIGS:
            d = time_loop(pipe, "DDIM", {}, 0.0, emb, lat, args.steps, 7.5, args.reps)
            v = time_loop(pipe, name, kw, eta, emb, lat, args.steps, 7.5, args.reps)
            ddim_pairs[name].append(d)
            runs[name].append(v)
    for name in runs:
        res["iter_per_s"][name] = {"runs": [round(v, 2) for v in runs[name]],
                                   "ddim_alternating": [round(v, 2) for v in ddim_pairs[name]],
                                   "ratio_to_ddim": round(float(np.median(runs[name]) / np.median(ddim_pairs[name])), 4)}
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()
