"""Host logic of the sigma-space samplers (EulerDiscrete, EulerAncestralDiscrete, LMSDiscrete) and DDIM with eta > 0:
the per-step plans against stateful twins written the way diffusers 0.30.2 steps (tests/sampler_twins.py), the
schedule pins, the closed-form identities that tie the samplers to DDIM, and the C layout of b200sd_sampler_coeffs."""
import ctypes
import os

import numpy as np
import pytest
import torch

import sampler_twins as T
from b200sd import scheduler as S
from oracle import restated as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIGMA_SCHEDULERS = ["EulerDiscrete", "EulerAncestralDiscrete", "LMSDiscrete"]
ABAR = torch.from_numpy(S.alphas_cumprod())  # the same fp32 table on both sides


def _eps_fn(seed):
    rng = np.random.RandomState(seed)
    w = rng.randn(2)

    def f(x_in, t):  # x_in: the UNet input (scaled sample)
        base = np.tanh(x_in * 0.7 + t / 1000.0)
        return base * w[0] + 0.1, base * w[1] - 0.05
    return f


def _noise(n_steps, shape, seed=7):
    rng = np.random.RandomState(seed)
    return [rng.randn(*shape) for _ in range(n_steps)]


@pytest.mark.parametrize("spacing", ["linspace", "leading", "trailing"])
def test_sigma_schedule_pins(spacing):
    s = S.EulerDiscreteScheduler(20, timestep_spacing=spacing)
    assert s.sigmas[-1] == 0.0 and len(s.sigmas) == 21
    train = np.sqrt((1 - s.abar) / s.abar)
    assert abs(train.max() - 14.614655) < 1e-6 and abs(train.min() - 0.029168) < 1e-6
    ts = s.timesteps
    assert all(isinstance(t, float) for t in ts) and len(ts) == 20
    if spacing == "linspace":
        assert ts[:3] == [999.0, 946.5, 894.0]
        assert np.allclose(s.sigmas[:3], [14.6147, 10.7469, 8.0815], atol=1e-4)
        assert abs(s.init_noise_sigma - 14.614655) < 1e-6
    elif spacing == "leading":
        assert ts[:3] == [951.0, 901.0, 851.0] and ts[-1] == 1.0
        assert abs(s.init_noise_sigma - 11.0736) < 1e-4
        assert abs(s.init_noise_sigma - np.sqrt(s.sigmas[0] ** 2 + 1)) < 1e-12
    else:
        assert ts[:3] == [999.0, 949.0, 899.0] and ts[-1] == 49.0
        assert abs(s.init_noise_sigma - 14.614655) < 1e-6
    # the UNet timestep is the fp16 value of the float timestep; the first input scale is c_in(sigma_0)
    tw = T.EulerTwin(20, ABAR, spacing)
    assert ts == [float(np.float16(t)) for t in tw.timesteps]
    assert np.allclose(s.sigmas, tw.sigmas.numpy(), rtol=1e-12, atol=0)
    assert abs(s.first_in_scale() - 1 / np.sqrt(s.sigmas[0] ** 2 + 1)) < 1e-15
    with pytest.raises(ValueError):
        S.EulerDiscreteScheduler(20, timestep_spacing="karras")


def test_reference_keys_registered_and_unknown_names_refused():
    for name in SIGMA_SCHEDULERS:
        assert name in S.SCHEDULER_MAP
    for bad in ("Euler", "EulerDiscreteScheduler", "LMS"):
        with pytest.raises(ValueError):
            S.make_scheduler(bad, 20)


def _run_plan_vs_twin(name, n, spacing, start=0, guidance=7.5):
    s = S.make_scheduler(name, n, timestep_spacing=spacing)
    tw = T.TWINS[name](n, ABAR, spacing, begin_index=start)
    f = _eps_fn(4)
    rng = np.random.RandomState(0)
    x = rng.randn(2, 4, 4) * s.init_noise_sigma
    noise = _noise(n + 1, x.shape)
    hist = [np.zeros_like(x) for _ in range(4)]
    xr = torch.from_numpy(x.copy())
    plan = s.plan(start=start)
    assert abs(s.first_in_scale(start) - float(1 / (tw.sigmas[start] ** 2 + 1) ** 0.5)) < 1e-15
    x_in = x * s.first_in_scale(start)
    for j, st in enumerate(plan):
        i = start + j
        assert st.timestep == tw.unet_timestep()
        assert np.allclose(x_in, tw.scale_model_input(xr).numpy(), rtol=1e-12, atol=1e-12)
        eu, ec = f(x_in, st.timestep)
        z = noise[st.noise_draw] if st.noise_scale else None
        x, x0, x_in = S.apply_plan_host(st, guidance, eu, ec, x, hist, noise=z, return_unet_in=True)
        e = torch.from_numpy(R.cfg_combine(eu, ec, guidance))
        xr, x0r = tw.step(e, xr, torch.from_numpy(noise[1 + j]))
        assert np.allclose(x, xr.numpy(), rtol=1e-8, atol=1e-8), (name, n, spacing, start, i)
        assert np.allclose(x0, x0r.numpy(), rtol=1e-8, atol=1e-8), (name, n, spacing, start, i)
    return plan


@pytest.mark.parametrize("name", SIGMA_SCHEDULERS)
@pytest.mark.parametrize("n", [4, 10, 20, 50])
def test_sampler_plans_match_twins(name, n):
    for spacing in ("linspace", "leading", "trailing"):
        plan = _run_plan_vs_twin(name, n, spacing)
        assert plan[-1].in_scale == 1.0  # the final sigma is 0
        if name == "EulerAncestralDiscrete":
            assert [p.noise_draw for p in plan] == list(range(1, n + 1)) and plan[-1].noise_scale == 0.0
        else:
            assert all(p.noise_scale == 0.0 for p in plan)


@pytest.mark.parametrize("name", SIGMA_SCHEDULERS)
@pytest.mark.parametrize("n,start", [(20, 10), (20, 3), (10, 5), (50, 25)])
def test_sampler_img2img_starts_match_fresh_twins(name, n, start):
    plan = _run_plan_vs_twin(name, n, "leading", start=start)
    if name == "LMSDiscrete":  # the derivative history starts empty at the start step
        assert plan[0].n_hist == 0 and plan[1].n_hist == 3
    s = S.make_scheduler(name, n, timestep_spacing="leading")
    x0, nz = np.full((1, 4, 2, 2), 2.0, np.float32), np.full((1, 4, 2, 2), -1.0, np.float32)
    strength = 1 - start / n
    k = s.start_step(strength)
    assert np.allclose(s.add_noise(x0, nz, strength), 2.0 - np.float32(s.sigmas[k]), rtol=1e-6)


@pytest.mark.parametrize("n", [4, 10, 20, 50])
@pytest.mark.parametrize("start", [0, 2])
def test_ddim_eta_matches_twin(n, start):
    eta = 0.7
    s = S.DDIMScheduler(n, eta=eta)
    s.abar = R.alphas_cumprod().double().numpy()
    tw = T.DDIMEtaTwin(n, R.alphas_cumprod(), eta)
    f = _eps_fn(5)
    rng = np.random.RandomState(1)
    x = rng.randn(2, 4, 4)
    noise = _noise(n + 1, x.shape)
    hist = [np.zeros_like(x) for _ in range(4)]
    xr = torch.from_numpy(x.copy())
    plan = s.plan(start=start)
    assert [p.timestep for p in plan] == tw.timesteps[start:] and s.uses_noise
    for j, st in enumerate(plan):
        eu, ec = f(x, st.timestep)
        x, x0 = S.apply_plan_host(st, 7.5, eu, ec, x, hist, noise=noise[st.noise_draw])
        xr, x0r = tw.step(torch.from_numpy(R.cfg_combine(eu, ec, 7.5)), st.timestep, xr, torch.from_numpy(noise[1 + j]))
        assert np.allclose(x, xr.numpy(), rtol=1e-8, atol=1e-8), (n, j)
        assert np.allclose(x0, x0r.numpy(), rtol=1e-8, atol=1e-8), (n, j)
    # eta = 0 keeps the deterministic coefficients exactly
    assert S.DDIMScheduler(n, eta=0.0).plan() == S.DDIMScheduler(n).plan()
    assert not S.DDIMScheduler(n).uses_noise
    with pytest.raises(ValueError):
        S.DDIMScheduler(n, eta=-1.0)


def _identity_run(n, name, eta):
    """Euler-type sampler and DDIM on leading timesteps, the same eps model of the UNet input, the same noise."""
    d = S.DDIMScheduler(n, eta=eta)
    e = S.make_scheduler(name, n, timestep_spacing="leading")
    assert [p.timestep for p in d.plan()] == [float(t) for t in e.timesteps]
    f = _eps_fn(6)
    rng = np.random.RandomState(2)
    xd = rng.randn(2, 4, 4)
    noise = _noise(n + 1, xd.shape)
    xe = xd * e.init_noise_sigma
    abar = d.abar
    hd = [np.zeros_like(xd) for _ in range(4)]
    he = [np.zeros_like(xd) for _ in range(4)]
    x_in_e = xe * e.first_in_scale()
    out = []
    for i, (sd, se) in enumerate(zip(d.plan(), e.plan())):
        t = int(sd.timestep)
        assert np.allclose(x_in_e, xd, rtol=1e-12, atol=1e-12)  # the UNet sees the DDIM variable
        eu, ec = f(xd, t)
        xd_new, x0d = S.apply_plan_host(sd, 7.5, eu, ec, xd, hd, noise=noise[sd.noise_draw] if sd.noise_scale else None)
        xe, x0e, x_in_e = S.apply_plan_host(se, 7.5, eu, ec, xe, he, return_unet_in=True,
                                            noise=noise[se.noise_draw] if se.noise_scale else None)
        assert np.allclose(x0e, x0d, rtol=1e-12, atol=1e-12)
        xd = xd_new
        if i + 1 < n:
            a_next = abar[int(d.plan()[i + 1].timestep)]
            out.append(float(np.abs(xe * np.sqrt(a_next) - xd).max()))
        else:
            out.append(float(np.abs(xe - x0d).max()))  # the last step lands on DDIM's x0
    return out


@pytest.mark.parametrize("n", [4, 10, 20, 50])
def test_euler_equals_ddim_eta0_in_the_scaled_variable(n):
    assert max(_identity_run(n, "EulerDiscrete", 0.0)) < 1e-12


@pytest.mark.parametrize("n", [4, 10, 20, 50])
def test_euler_ancestral_equals_ddim_eta1_under_the_same_noise(n):
    assert max(_identity_run(n, "EulerAncestralDiscrete", 1.0)) < 1e-12


@pytest.mark.parametrize("spacing", ["linspace", "leading", "trailing"])
def test_lms_coefficients(spacing):
    s = S.LMSDiscreteScheduler(20, timestep_spacing=spacing)
    tw = T.LMSTwin(20, ABAR, spacing)
    sig = s.sigmas
    for i in range(20):
        order = min(i + 1, 4)
        c = S.lms_coefficients(sig, i, order)
        # the weights of one step sum to the interval length (a constant derivative is integrated exactly)
        assert abs(sum(c) - (sig[i + 1] - sig[i])) < 1e-12 * max(1.0, abs(sig[i + 1] - sig[i]))
        # scipy.integrate.quad of the Lagrange basis
        q = [tw.lms_coefficient(order, i, k) for k in range(order)]
        assert np.allclose(c, q, rtol=1e-12, atol=1e-12), (i, c, q)
        # a derivative that is a polynomial of degree order-1 in sigma is integrated exactly
        rng = np.random.RandomState(i)
        poly = rng.randn(order)
        d = lambda v: np.polyval(poly, v)  # noqa: E731
        exact = np.polyval(np.polyint(poly), sig[i + 1]) - np.polyval(np.polyint(poly), sig[i])
        got = sum(ck * d(sig[i - k]) for k, ck in enumerate(c))
        assert abs(got - exact) < 1e-9 * max(1.0, abs(exact)), (i, got, exact)


def test_lms_step_is_exact_for_a_cubic_derivative():
    """Drive the LMS plan with eps = p(sigma), p a cubic: from the fourth step on, x_{i+1} - x_i is the exact integral."""
    s = S.LMSDiscreteScheduler(20, timestep_spacing="leading")
    poly = np.array([0.01, -0.2, 0.5, 1.5])
    sig = s.sigmas
    x = np.zeros(3)
    hist = [np.zeros_like(x) for _ in range(4)]
    for j, st in enumerate(s.plan()):
        e = np.full(3, np.polyval(poly, sig[j]))
        xn, _ = S.apply_plan_host(st, 1.0, np.zeros(3), e, x, hist)
        if j >= 3:
            ip = np.polyint(poly)
            exact = np.polyval(ip, sig[j + 1]) - np.polyval(ip, sig[j])
            assert np.allclose(xn - x, exact, rtol=1e-9, atol=1e-9), j
        x = xn


def test_lms_product_does_not_import_scipy():
    import subprocess
    import sys
    code = ("import sys; from b200sd import scheduler as S; S.LMSDiscreteScheduler(20).plan(); "
            "assert 'scipy' not in sys.modules, 'scipy imported'")
    subprocess.run([sys.executable, "-c", code], check=True, cwd=ROOT)


def test_apply_plan_host_noise_and_input_scale():
    st = S.EulerAncestralDiscreteScheduler(10).plan()[0]
    x = np.ones(4)
    with pytest.raises(ValueError, match="noise"):
        S.apply_plan_host(st, 1.0, np.zeros(4), np.zeros(4), x, [None] * 4)
    xp, x0, x_in = S.apply_plan_host(st, 1.0, np.zeros(4), np.zeros(4), x, [None] * 4, noise=np.full(4, 2.0),
                                     return_unet_in=True)
    assert np.allclose(xp, 1.0 + 2.0 * st.noise_scale) and np.allclose(x_in, st.in_scale * xp)


def test_sampler_coeffs_layout_matches_header(tmp_path):
    """sizeof / offsetof of b200sd_sampler_coeffs as gcc sees include/b200sd.h == the ctypes mirror in lib.py."""
    import shutil
    import subprocess

    from b200sd import lib
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    fields = [f[0] for f in lib.SamplerCoeffs._fields_]
    src = ['#include <stdio.h>', '#include <stddef.h>', '#include "b200sd.h"', 'int main(void) {',
           'printf("%zu\\n", sizeof(b200sd_sampler_coeffs));']
    src += [f'printf("%zu\\n", offsetof(b200sd_sampler_coeffs, {f}));' for f in fields]
    src += ['printf("%zu\\n", offsetof(b200sd_sampler_coeffs, step.noise_pred_nhwc));', 'return 0; }']
    c = tmp_path / "layout.c"
    c.write_text("\n".join(src))
    exe = tmp_path / "layout"
    subprocess.run([gcc, "-I", os.path.join(ROOT, "include"), str(c), "-o", str(exe)], check=True)
    vals = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = [ctypes.sizeof(lib.SamplerCoeffs)] + [getattr(lib.SamplerCoeffs, f).offset for f in fields]
    want += [lib.StepCoeffs.noise_pred_nhwc.offset]
    assert vals == want
    assert "b200sd_sampler_step" in lib.EXPORTED_SYMBOLS
