"""Stateful restatements of the diffusers 0.30.2 sigma-space samplers and of DDIM with eta > 0, written the way those
schedulers step (a per-call step index, a list of derivatives, LMS coefficients from ``scipy.integrate.quad``), to
check the per-step linear plans of ``b200sd.scheduler`` against.  float64 torch on the CPU; test-side only."""
from __future__ import annotations

import numpy as np
import torch


def _sigma_schedule(abar, n, spacing, steps_offset, n_train=1000):
    if spacing == "linspace":
        ts = np.linspace(0, n_train - 1, n, dtype=np.float32)[::-1].copy()
    elif spacing == "leading":
        ratio = n_train // n
        ts = (np.arange(0, n) * ratio).round()[::-1].copy().astype(np.float32) + steps_offset
    elif spacing == "trailing":
        ratio = n_train / n
        ts = np.arange(n_train, 0, -ratio).round().copy().astype(np.float32) - 1
    else:
        raise ValueError(spacing)
    sig = ((1 - abar) / abar) ** 0.5
    sig = np.interp(ts.astype(np.float64), np.arange(0, len(sig)), sig.numpy())
    return ts, torch.from_numpy(np.concatenate([sig, [0.0]]))


class _SigmaTwin:
    def __init__(self, n, abar, timestep_spacing="linspace", steps_offset=1, begin_index=0):
        self.abar = abar.double()
        self.timesteps, self.sigmas = _sigma_schedule(self.abar, n, timestep_spacing, steps_offset)
        smax = self.sigmas.max()
        self.init_noise_sigma = float(smax if timestep_spacing in ("linspace", "trailing") else (smax ** 2 + 1) ** 0.5)
        self.step_index = begin_index

    def scale_model_input(self, sample):
        return sample / ((self.sigmas[self.step_index] ** 2 + 1) ** 0.5)

    def unet_timestep(self):
        return float(np.float16(self.timesteps[self.step_index]))


class EulerTwin(_SigmaTwin):
    def step(self, model_output, sample, noise=None):
        sigma = self.sigmas[self.step_index]
        pred_original_sample = sample - sigma * model_output
        derivative = (sample - pred_original_sample) / sigma
        dt = self.sigmas[self.step_index + 1] - sigma
        self.step_index += 1
        return sample + derivative * dt, pred_original_sample


class EulerAncestralTwin(_SigmaTwin):
    def step(self, model_output, sample, noise):
        sigma = self.sigmas[self.step_index]
        pred_original_sample = sample - sigma * model_output
        sigma_from, sigma_to = sigma, self.sigmas[self.step_index + 1]
        sigma_up = (sigma_to ** 2 * (sigma_from ** 2 - sigma_to ** 2) / sigma_from ** 2) ** 0.5
        sigma_down = (sigma_to ** 2 - sigma_up ** 2) ** 0.5
        derivative = (sample - pred_original_sample) / sigma
        prev_sample = sample + derivative * (sigma_down - sigma)
        prev_sample = prev_sample + noise * sigma_up
        self.step_index += 1
        return prev_sample, pred_original_sample


class LMSTwin(_SigmaTwin):
    """order 4; the derivative list starts empty at ``begin_index`` (image-to-image: a loop that starts part-way)."""

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self.derivatives = []

    def lms_coefficient(self, order, t, current_order):
        from scipy import integrate

        sig = self.sigmas.numpy()

        def lms_derivative(tau):
            prod = 1.0
            for k in range(order):
                if current_order == k:
                    continue
                prod *= (tau - sig[t - k]) / (sig[t - current_order] - sig[t - k])
            return prod

        return integrate.quad(lms_derivative, sig[t], sig[t + 1], epsrel=1e-13, epsabs=1e-15)[0]

    def step(self, model_output, sample, noise=None, order=4):
        sigma = self.sigmas[self.step_index]
        pred_original_sample = sample - sigma * model_output
        derivative = (sample - pred_original_sample) / sigma
        self.derivatives.append(derivative)
        if len(self.derivatives) > order:
            self.derivatives.pop(0)
        order = min(len(self.derivatives), order)
        coeffs = [self.lms_coefficient(order, self.step_index, k) for k in range(order)]
        prev_sample = sample + sum(c * d for c, d in zip(coeffs, reversed(self.derivatives)))
        self.step_index += 1
        return prev_sample, pred_original_sample


class DDIMEtaTwin:
    """DDIMScheduler.step with eta (leading spacing, steps_offset 1, set_alpha_to_one False)."""

    def __init__(self, n, abar, eta, steps_offset=1, n_train=1000):
        self.abar = abar.double()
        self.n, self.eta, self.ratio = n, eta, n_train // n
        self.timesteps = [i * self.ratio + steps_offset for i in range(n)][::-1]

    def step(self, model_output, t, sample, noise):
        prev_t = t - self.ratio
        a_t = self.abar[t]
        a_p = self.abar[prev_t] if prev_t >= 0 else self.abar[0]
        pred_original_sample = (sample - (1 - a_t) ** 0.5 * model_output) / a_t ** 0.5
        variance = (1 - a_p) / (1 - a_t) * (1 - a_t / a_p)
        std_dev_t = self.eta * variance ** 0.5
        prev_sample = a_p ** 0.5 * pred_original_sample + (1 - a_p - std_dev_t ** 2) ** 0.5 * model_output
        if self.eta > 0:
            prev_sample = prev_sample + std_dev_t * noise
        return prev_sample, pred_original_sample


TWINS = {"EulerDiscrete": EulerTwin, "EulerAncestralDiscrete": EulerAncestralTwin, "LMSDiscrete": LMSTwin}
