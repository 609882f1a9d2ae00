"""GPU tests of the sampler step (b200sd_sampler_step) and of the EulerDiscrete, EulerAncestralDiscrete, LMSDiscrete and
DDIM eta > 0 samplers in the device loop: the kernel against its numpy mirror and the Philox twin, the loop graph against
a host loop of the stateful twins on the oracle UNet, graph == eager, seeds, and full-size SD-2.1-base runs."""
import numpy as np
import pytest
import torch

import sampler_twins as T
from b200sd import config
from b200sd import scheduler as S
from b200sd.rng import NvRandomSource
from oracle import restated as R

pytestmark = pytest.mark.gpu

NEW = ["EulerDiscrete", "EulerAncestralDiscrete", "LMSDiscrete"]
ALL = [("DDIM", {}), ("DDIM", {"eta": 0.8}), ("DPMSolverMultistep", {}), ("PNDM", {}), ("EulerDiscrete", {}),
       ("EulerAncestralDiscrete", {"timestep_spacing": "leading"}), ("LMSDiscrete", {"timestep_spacing": "trailing"})]


def _philox(seed, draw, count):
    src = NvRandomSource(seed)
    src.offset = draw
    return src.normal_array(count).astype(np.float32)


def _key(seed):
    return torch.from_numpy(np.array([seed & 0xFFFFFFFF, 0], dtype=np.uint32).view(np.int32)).cuda()


def _sampler_coeffs(lib, st, g, n, nhwc):
    k = lib.SamplerCoeffs()
    k.step.guidance = g
    k.step.cx, k.step.ce, k.step.x0_cx, k.step.x0_ce = st.cx, st.ce, st.x0_cx, st.x0_ce
    for j in range(4):
        k.step.ch[j], k.step.x0_ch[j] = st.ch[j], st.x0_ch[j]
    k.step.n_hist, k.step.push_eps_slot, k.step.push_x0_slot, k.step.push_x_slot = (st.n_hist, st.push_eps_slot,
                                                                                    st.push_x0_slot, st.push_x_slot)
    k.step.noise_pred_nhwc = int(nhwc)
    k.in_scale, k.noise_scale, k.noise_draw = st.in_scale, st.noise_scale, n * st.noise_draw
    return k


@pytest.mark.parametrize("nhwc", [False, True])
@pytest.mark.parametrize("name,kw", ALL)
def test_sampler_step_matches_host_mirror(cuda_lib, name, kw, nhwc):
    lib = cuda_lib
    n, c, h, w, c_pad, seed, g = 2, 4, 16, 16, 8, 1234, 6.0
    sched = S.make_scheduler(name, 10, **kw)
    gen = torch.Generator().manual_seed(5)
    x = torch.randn(n, c, h, w, generator=gen) * 3
    hist = torch.randn(4, n, c, h, w, generator=gen)
    for st in sched.plan()[:4]:
        eps = torch.randn(2 * n, c, h, w, generator=gen)
        z = None
        if st.noise_scale:
            z = np.stack([_philox(seed, n * st.noise_draw + b, c * h * w).reshape(c, h, w) for b in range(n)])
        hh = [hist[j].double().numpy().copy() for j in range(4)]
        xp, x0, x_in = S.apply_plan_host(st, g, eps[:n].double().numpy(), eps[n:].double().numpy(), x.double().numpy(),
                                         hh, noise=z, return_unet_in=True)
        lat, den, hd = x.cuda(), torch.empty(n, c, h, w, device="cuda"), hist.cuda()
        unet_in = torch.full((2 * n, h, w, c_pad), 0.0, dtype=torch.float16, device="cuda")
        ep = (eps.permute(0, 2, 3, 1) if nhwc else eps).contiguous().cuda()
        lib.sampler_step(ep, lat, _sampler_coeffs(lib, st, g, n, nhwc), hist=hd, denoised=den, unet_in=unet_in,
                         rng_key=_key(seed))
        scale = max(1.0, float(np.abs(xp).max()))
        assert np.abs(lat.cpu().double().numpy() - xp).max() < 2e-5 * scale, (name, kw)
        assert np.abs(den.cpu().double().numpy() - x0).max() < 2e-5 * max(1.0, float(np.abs(x0).max()))
        for j in range(4):
            assert np.abs(hd[j].cpu().double().numpy() - hh[j]).max() < 2e-5 * max(1.0, float(np.abs(hh[j]).max()))
        want = torch.from_numpy(x_in).float().permute(0, 2, 3, 1)
        got = unet_in.cpu().float()
        tol = 2e-3 * want.abs() + 1e-3
        assert ((got[:n, ..., :c] - want).abs() <= tol).all() and ((got[n:, ..., :c] - want).abs() <= tol).all()
        assert (got[..., c:] == 0).all()  # padding channels untouched


def test_sampler_step_extension_off_is_the_plain_step_bit_for_bit(cuda_lib):
    lib = cuda_lib
    n, c, h, w = 2, 4, 24, 24
    gen = torch.Generator(device="cuda").manual_seed(9)
    for st in S.PNDMScheduler(10).plan()[:5] + S.DDIMScheduler(10).plan()[:2]:
        eps = torch.randn(2 * n, c, h, w, device="cuda", generator=gen)
        x = torch.randn(n, c, h, w, device="cuda", generator=gen)
        hist = torch.randn(4, n, c, h, w, device="cuda", generator=gen)
        outs = []
        for new in (False, True):
            lat, hd, den = x.clone(), hist.clone(), torch.empty_like(x)
            ui = torch.zeros(2 * n, h, w, 8, dtype=torch.float16, device="cuda")
            k = _sampler_coeffs(lib, st, 7.5, n, False)
            if new:
                lib.sampler_step(eps, lat, k, hist=hd, denoised=den, unet_in=ui)
            else:
                lib.cfg_scheduler_step(eps, lat, k.step, hist=hd, denoised=den, unet_in=ui)
            outs.append((lat, hd, den, ui))
        for a, b in zip(*outs):
            assert torch.equal(a, b)


def test_device_noise_matches_the_nvidia_rng_twin(cuda_lib):
    """cx = ce = 0, noise_scale = 1: the kernel writes its Philox normals; compare with rng.NvRandomSource draws."""
    lib = cuda_lib
    n, c, h, w = 3, 4, 64, 64
    per = c * h * w
    for seed, draw in ((0, 0), (42, 5), (2 ** 32 - 1, 1000)):
        k = lib.SamplerCoeffs()
        k.noise_scale, k.noise_draw, k.in_scale = 1.0, draw, 1.0
        k.step.push_eps_slot = k.step.push_x0_slot = k.step.push_x_slot = -1
        lat = torch.zeros(n, c, h, w, device="cuda")
        lib.sampler_step(torch.zeros(2 * n, c, h, w, device="cuda"), lat, k, rng_key=_key(seed))
        got = lat.cpu().numpy().reshape(n, per)
        want = np.stack([_philox(seed, draw + b, per) for b in range(n)])
        assert np.abs(got - want).max() <= 1e-6
        assert (got == want).mean() >= 0.999, (got == want).mean()
    # the initial latents of prepare_latents(rng="nvidia") are draws 0 .. n-1 of the same stream
    from b200sd.pipeline import B200StableDiffusionPipeline
    import types
    stub = types.SimpleNamespace(vae_scale_factor=8)
    lat0 = B200StableDiffusionPipeline.prepare_latents(stub, 2, 4, 128, 128, seed=77, rng="nvidia")
    assert np.array_equal(lat0.reshape(2, -1), np.stack([_philox(77, b, 4 * 16 * 16) for b in range(2)]))


def test_sampler_step_input_only_mode(cuda_lib):
    lib = cuda_lib
    n, c, h, w = 2, 4, 16, 16
    x = torch.randn(n, c, h, w, device="cuda")
    k = lib.SamplerCoeffs()
    k.in_scale = 0.0683
    ui = torch.zeros(2 * n, h, w, 8, dtype=torch.float16, device="cuda")
    lat = x.clone()
    lib.sampler_step(None, lat, k, unet_in=ui)
    want = (x * np.float32(0.0683)).half().permute(0, 2, 3, 1)
    assert torch.equal(ui[:n, ..., :c], want) and torch.equal(ui[n:, ..., :c], want)
    assert (ui[..., c:] == 0).all() and torch.equal(lat, x)
    with pytest.raises(lib.B200SDError):
        lib.sampler_step(None, lat, k)


# ---------------------------------------------------------------- tiny UNet loops
def _tiny(name, seed=31, **kw):
    from b200sd.pipeline import B200StableDiffusionPipeline
    pipe = B200StableDiffusionPipeline.from_random_init("tiny", images_per_call=1, height=64, width=64, seed=seed, **kw)
    return pipe


def _with_scheduler(pipe, name, **kw):
    pipe.scheduler_name = name
    pipe.scheduler_kwargs = dict(kw)
    return pipe


@pytest.mark.parametrize("name,spacing", [("EulerDiscrete", "linspace"), ("EulerAncestralDiscrete", "leading"),
                                          ("LMSDiscrete", "linspace"), ("LMSDiscrete", "trailing")])
def test_tiny_loop_vs_twin_oracle_loop(cuda_lib, name, spacing):
    pipe = _with_scheduler(_tiny(name), name, timestep_spacing=spacing)
    steps, g, seed = 6, 5.0, 4321
    sched = pipe._make_scheduler(steps)
    np.random.seed(3)
    lat0 = np.random.randn(1, 4, 16, 16).astype(np.float16).astype(np.float32) * np.float32(sched.init_noise_sigma)
    emb = pipe._encode_prompt(["a red cube"], True, None)
    final = pipe.denoise(emb, lat0, steps, g, seed=seed).cpu().clone()
    # graph == eager, bit for bit
    rec = []
    eager = pipe.denoise(emb, lat0, steps, g, record=rec, seed=seed).cpu().clone()
    assert torch.equal(final, eager), float((final - eager).abs().max())
    assert [r[0] for r in rec] == sched.timesteps
    # the same seed twice: the same latents
    assert torch.equal(final, pipe.denoise(emb, lat0, steps, g, seed=seed).cpu())
    # oracle loop: the stateful twin on the oracle UNet, the same Philox draws
    usd = config.random_state_dict(config.unet_param_shapes(config.TINY_UNET), seed=31, dtype=torch.float16)
    tw = T.TWINS[name](steps, torch.from_numpy(S.alphas_cumprod()), spacing)
    x = torch.from_numpy(lat0).double()
    embt = torch.from_numpy(emb).float()
    with torch.no_grad():
        for j in range(steps):
            xin = tw.scale_model_input(x).float()
            t = tw.unet_timestep()
            eps = R.unet_forward(usd, config.TINY_UNET, torch.cat([xin, xin]).half().float(), torch.tensor([t] * 2), embt)
            z = torch.from_numpy(_philox(seed, 1 + j, 4 * 16 * 16).reshape(1, 4, 16, 16)).double()
            x, _ = tw.step(R.cfg_combine(eps[:1], eps[1:], g).double(), x, z)
    rel = float((final.double() - x).abs().max() / x.abs().max())
    print(f"{name} ({spacing}): latent rel err after {steps} steps = {rel:.3e}")
    assert rel < 3e-2
    if name == "EulerAncestralDiscrete":  # another seed, another image
        other = pipe.denoise(emb, lat0, steps, g, seed=seed + 1).cpu()
        assert not torch.allclose(other, final)


def test_tiny_euler_ancestral_equals_ddim_eta1_on_the_device(cuda_lib):
    """Leading spacing: the UNet sees the DDIM variable, the noise is the same Philox stream, so the denoised estimates
    of the two loops agree (up to fp16 rounding of the UNet input)."""
    pipe = _tiny("DDIM")
    steps, g, seed = 6, 5.0, 99
    np.random.seed(4)
    lat_d = np.random.randn(1, 4, 16, 16).astype(np.float16).astype(np.float32)
    emb = pipe._encode_prompt(["a blue sphere"], True, None)
    _with_scheduler(pipe, "DDIM")
    x0_ddim = pipe.denoise(emb, lat_d, steps, g, eta=1.0, seed=seed, return_denoised=True).cpu().clone()
    lat_ddim = pipe._latents.cpu().clone()
    _with_scheduler(pipe, "EulerAncestralDiscrete", timestep_spacing="leading")
    sched = pipe._make_scheduler(steps)
    x0_ea = pipe.denoise(emb, lat_d * np.float32(sched.init_noise_sigma), steps, g, seed=seed,
                         return_denoised=True).cpu().clone()
    rel = float((x0_ea - x0_ddim).abs().max() / x0_ddim.abs().max())
    print(f"Euler-ancestral vs DDIM eta=1: x0 rel err = {rel:.3e}")
    assert rel < 1e-2
    # and eta = 1 is not eta = 0
    _with_scheduler(pipe, "DDIM")
    assert not torch.allclose(pipe.denoise(emb, lat_d, steps, g, seed=seed).cpu(), lat_ddim)


def test_tiny_img2img_and_controlnet_with_euler(cuda_lib):
    # image-to-image: sigma-space noising, the loop from the start step; graph == eager
    pipe = _with_scheduler(_tiny("EulerDiscrete", with_vae_encoder=True), "EulerDiscrete")
    img0 = (torch.rand(1, 3, 64, 64, generator=torch.Generator().manual_seed(32)) * 2 - 1).half().numpy()
    kw = dict(height=64, width=64, num_inference_steps=8, guidance_scale=6.0, starting_image=img0, strength=0.5,
              output_type="np")
    np.random.seed(33)
    a = pipe("a cat", **kw).images
    pipe.loop_graph = False
    np.random.seed(33)
    b = pipe("a cat", **kw).images
    pipe.loop_graph = True
    assert a.shape == (1, 64, 64, 3) and np.isfinite(a).all() and np.array_equal(a, b)
    sched = pipe._make_scheduler(8)
    assert sched.start_step(0.5) == 4
    # ControlNet + Euler: the ControlNets read the scaled UNet input; graph == eager
    pipe = _with_scheduler(_tiny("EulerDiscrete", seed=21, controlnet_cfgs=[config.TINY_CONTROLNET]), "EulerDiscrete")
    np.random.seed(5)
    lat0 = np.random.randn(1, 4, 16, 16).astype(np.float16).astype(np.float32) * np.float32(14.614655)
    cond = np.random.rand(3, 128, 128).astype(np.float16)
    cc = pipe.prepare_control_cond([cond], True, 1, 1)
    emb = pipe._encode_prompt(["a cat"], True, None)
    g_out = pipe.denoise(emb, lat0, 3, 5.0, controlnet_cond=cc).cpu().clone()
    e_out = pipe.denoise(emb, lat0, 3, 5.0, controlnet_cond=cc, record=[]).cpu().clone()
    assert torch.isfinite(g_out).all() and torch.equal(g_out, e_out)


def test_call_surface(cuda_lib):
    """__call__: eta reaches DDIM only; seeds reproduce ancestral images; a negative eta is refused."""
    pipe = _tiny("DDIM")
    kw = dict(height=64, width=64, num_inference_steps=4, guidance_scale=5.0, output_type="np", seed=11, rng="nvidia")
    a = pipe("a cat", eta=0.5, **kw).images
    assert np.array_equal(a, pipe("a cat", eta=0.5, **kw).images)
    assert not np.array_equal(a, pipe("a cat", **kw).images)
    with pytest.raises(ValueError):
        pipe("a cat", eta=-1.0, **kw)
    _with_scheduler(pipe, "EulerAncestralDiscrete")
    b = pipe("a cat", **kw).images
    assert np.array_equal(b, pipe("a cat", **kw).images)
    assert not np.array_equal(b, pipe("a cat", **dict(kw, seed=12)).images)
    # eta is ignored by the samplers that do not take it, like the reference
    _with_scheduler(pipe, "EulerDiscrete")
    assert np.array_equal(pipe("a cat", eta=0.3, **kw).images, pipe("a cat", **kw).images)


def test_from_pretrained_with_a_sampler_override(cuda_lib, tmp_path):
    import json
    import os
    st = pytest.importorskip("safetensors.torch")
    from b200sd.pipeline import B200StableDiffusionPipeline
    ucfg, vcfg = config.TINY_UNET, config.TINY_VAE
    for name, sd, cfg in (("unet", config.random_state_dict(config.unet_param_shapes(ucfg), seed=3, dtype=torch.float16), ucfg),
                          ("vae", config.random_state_dict(config.vae_decoder_param_shapes(vcfg), seed=4, dtype=torch.float16), vcfg)):
        os.makedirs(tmp_path / name)
        st.save_file({k: v.contiguous() for k, v in sd.items()}, str(tmp_path / name / "diffusion_pytorch_model.safetensors"))
        (tmp_path / name / "config.json").write_text(json.dumps({k: (list(v) if isinstance(v, tuple) else v) for k, v in cfg.items()}))
    os.makedirs(tmp_path / "scheduler")
    (tmp_path / "scheduler" / "scheduler_config.json").write_text(json.dumps(
        {"_class_name": "EulerDiscreteScheduler", "timestep_spacing": "leading", "steps_offset": 1}))
    pipe = B200StableDiffusionPipeline.from_pretrained(str(tmp_path), height=64, width=64,
                                                       scheduler_override="EulerDiscrete")
    assert pipe.scheduler_name == "EulerDiscrete"
    assert pipe.scheduler_kwargs == {"timestep_spacing": "leading", "steps_offset": 1}
    img = pipe("a cat", height=64, width=64, num_inference_steps=3, output_type="np", seed=1).images
    assert np.isfinite(img).all()


# ---------------------------------------------------------------- SD-2.1-base 512x512
@pytest.fixture(scope="module")
def sd21(cuda_lib):
    from b200sd.pipeline import B200StableDiffusionPipeline
    return B200StableDiffusionPipeline.from_random_init("sd21-base", images_per_call=1, height=512, width=512, seed=0)


@pytest.mark.parametrize("name", NEW)
def test_sd21_base_512_twenty_steps(sd21, name):
    pipe = _with_scheduler(sd21, name)
    steps, g, seed = 20, 7.5, 5
    sched = pipe._make_scheduler(steps)
    np.random.seed(0)
    lat0 = np.random.randn(1, 4, 64, 64).astype(np.float16).astype(np.float32) * np.float32(sched.init_noise_sigma)
    emb = pipe._encode_prompt(["a photo of an astronaut riding a horse"], True, None)
    final = pipe.denoise(emb, lat0, steps, g, seed=seed).cpu().clone()
    assert torch.isfinite(final).all()
    eager = pipe.denoise(emb, lat0, steps, g, seed=seed, record=[]).cpu()
    assert torch.equal(final, eager), float((final - eager).abs().max())
    out = pipe("a photo of an astronaut riding a horse", num_inference_steps=steps, guidance_scale=g, output_type="np",
               seed=seed)
    assert out.images.shape == (1, 512, 512, 3) and np.isfinite(out.images).all()
