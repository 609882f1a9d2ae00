"""Host side of the fused CFG + scheduler-step kernel: per-step fp32 coefficients.

The reference does this math on the host, per element, in fp32: Python defers to diffusers
(``pipeline.py:475-476,504-505,565-569``), the in-tree spec is the Swift twin
(``swift/StableDiffusion/pipeline/Scheduler.swift:137-344`` PNDM/PLMS,
``DPMSolverMultistepScheduler.swift:27-245`` DPM-Solver++ 2M; DDIM == its first-order update,
``:153-174``).  Every one of those updates is *linear* in (x_t, eps, history), so here each
scheduler only produces, per step, the scalars of

    x_prev = cx * x + ce * eps + sum_i ch[i]    * hist[i]
    x0     = x0_cx * x + x0_ce * eps + sum_i x0_ch[i] * hist[i]

plus which history slots to overwrite; ``b200sd_cfg_scheduler_step`` applies them on the device
(one launch, also does classifier-free guidance and writes the next UNet input), so the denoising
loop never synchronises with the host.  Coefficients are computed in float64 and rounded once.

The sigma-space samplers of diffusers 0.30.2 (EulerDiscrete, EulerAncestralDiscrete, LMSDiscrete), which the
reference's Python pipeline offers (``pipeline.py:592-604``), and DDIM with eta > 0 add three per-step terms that the
same kernel (``b200sd_sampler_step``) applies: ``in_scale``, the NEXT step's ``c_in = 1 / sqrt(sigma^2 + 1)``
(``scale_model_input``, pipeline.py:504-508) on the value written as the next UNet input; ``noise_scale`` times a
Philox normal drawn on the device (Euler-ancestral ``sigma_up``, DDIM's ``std_dev_t``); and ``noise_draw``, which block
of that Philox stream the step uses (image ``b`` of ``n`` draws ``n * noise_draw + b``; draws ``0 .. n-1`` are the
initial latents of ``rng="nvidia"``).
"""
from __future__ import annotations

import dataclasses
import math
from typing import List

import numpy as np


@dataclasses.dataclass
class StepPlan:
    """One denoising step: UNet timestep + the linear-update coefficients (+ the sampler terms, see the module doc)."""
    timestep: float
    cx: float
    ce: float
    ch: List[float]
    x0_cx: float
    x0_ce: float
    x0_ch: List[float]
    n_hist: int = 0
    push_eps_slot: int = -1
    push_x0_slot: int = -1
    push_x_slot: int = -1
    in_scale: float = 1.0
    noise_scale: float = 0.0
    noise_draw: int = 0


def alphas_cumprod(beta_start=0.00085, beta_end=0.012, n=1000, schedule="scaled_linear"):
    """fp32 like the reference (Scheduler.swift:168-186)."""
    if schedule == "scaled_linear":
        betas = np.linspace(np.float32(beta_start) ** 0.5, np.float32(beta_end) ** 0.5, n, dtype=np.float32) ** 2
    elif schedule == "linear":
        betas = np.linspace(beta_start, beta_end, n, dtype=np.float32)
    else:
        raise ValueError(f"unknown beta schedule {schedule}")
    return np.cumprod((1.0 - betas).astype(np.float32), dtype=np.float32)


class _Base:
    init_noise_sigma = 1.0
    n_hist_slots = 4

    def __init__(self, num_inference_steps, num_train_timesteps=1000, beta_start=0.00085, beta_end=0.012,
                 beta_schedule="scaled_linear"):
        if num_inference_steps < 1:
            raise ValueError("num_inference_steps must be >= 1")
        self.n = int(num_inference_steps)
        self.n_train = int(num_train_timesteps)
        self.abar = alphas_cumprod(beta_start, beta_end, num_train_timesteps, beta_schedule).astype(np.float64)

    def scale_model_input(self, x, t):  # identity for DDIM / PNDM / DPM (pipeline.py:504)
        return x

    def first_in_scale(self, start: int = 0) -> float:
        """Scale of the first UNet input of a loop that starts at ``start`` (the later ones are ``StepPlan.in_scale``)."""
        return 1.0

    @property
    def uses_noise(self) -> bool:
        return False

    @property
    def timesteps(self):
        return [p.timestep for p in self.plan()]

    def plan(self, start: int = 0) -> List[StepPlan]:
        """Steps ``start`` .. end of the schedule, with the multistep state starting empty at ``start`` (what a
        fresh Swift scheduler does when the pipeline feeds it ``calculateTimesteps(strength)``)."""
        raise NotImplementedError

    # ---- image-to-image (Scheduler.swift:83-114) ----
    def start_step(self, strength: float) -> int:
        """max(inferenceStepCount - Int(Float(inferenceStepCount) * strength), 0)."""
        return max(self.n - int(np.float32(self.n) * np.float32(strength)), 0)

    def calculate_timesteps(self, strength=None):
        ts = self.timesteps
        return ts if strength is None else ts[self.start_step(strength):]

    def add_noise(self, original_sample, noise, strength):
        """sqrt(abar_t) * x0 + sqrt(1 - abar_t) * noise at t = timeSteps[startStep]."""
        t = self.timesteps[self.start_step(strength)]
        a = np.float32(self.abar[t])
        return np.float32(np.sqrt(a)) * original_sample + np.float32(np.sqrt(np.float32(1.0) - a)) * noise


class DDIMScheduler(_Base):
    """Epsilon prediction, 'leading' spacing, steps_offset 1, set_alpha_to_one False.  ``eta`` > 0 adds
    ``std_dev_t = eta * sqrt((1 - a_p) / (1 - a_t) * (1 - a_t / a_p))`` times fresh noise and takes ``std_dev_t^2`` out
    of the direction term (diffusers 0.30.2 ``DDIMScheduler.step``); eta = 0 is the deterministic update."""

    def __init__(self, num_inference_steps, steps_offset=1, eta=0.0, **kw):
        super().__init__(num_inference_steps, **kw)
        self.steps_offset = steps_offset
        self.eta = float(eta)
        if self.eta < 0:
            raise ValueError(f"eta must be >= 0, got {eta}")

    @property
    def uses_noise(self):
        return self.eta != 0.0

    def plan(self, start=0):
        ratio = self.n_train // self.n
        ts = [int(round(i * ratio)) + self.steps_offset for i in range(self.n)][::-1]
        out = []
        for j, t in enumerate(ts[start:]):
            tp = t - ratio
            a_t = self.abar[t]
            a_p = self.abar[tp] if tp >= 0 else self.abar[0]
            x0_cx = 1.0 / math.sqrt(a_t)
            x0_ce = -math.sqrt(1 - a_t) / math.sqrt(a_t)
            cx = math.sqrt(a_p) * x0_cx
            if self.eta == 0.0:
                ce = math.sqrt(a_p) * x0_ce + math.sqrt(1 - a_p)
                out.append(StepPlan(t, cx, ce, [0.0] * 4, x0_cx, x0_ce, [0.0] * 4))
                continue
            std = self.eta * math.sqrt((1 - a_p) / (1 - a_t) * (1 - a_t / a_p))
            ce = math.sqrt(a_p) * x0_ce + math.sqrt(max(1 - a_p - std * std, 0.0))
            out.append(StepPlan(t, cx, ce, [0.0] * 4, x0_cx, x0_ce, [0.0] * 4, noise_scale=std, noise_draw=1 + j))
        return out


class DPMSolverMultistepScheduler(_Base):
    """DPM-Solver++(2M) midpoint, epsilon prediction, 'linspace' spacing; first step and (for < 15
    steps) the last two steps are first order (DPMSolverMultistepScheduler.swift:216-244).
    History ring: x0 of the previous step in slots 0/1.

    ``final_sigmas_type``: how the LAST step ends.  ``"sigma_min"``: at the first training timestep's (alpha, sigma),
    what the in-tree Swift scheduler does (``alpha_t[0] / sigma_t[0]``, DPMSolverMultistepScheduler.swift:214-222).
    ``"zero"``: diffusers 0.30.2's default, which the reference's PYTHON pipeline runs (pipeline.py:565-569 ->
    ``scheduler.step``): the final sigma is 0, the last step is always first order and lands exactly on the
    denoised estimate x0."""

    def __init__(self, num_inference_steps, final_sigmas_type="sigma_min", **kw):
        super().__init__(num_inference_steps, **kw)
        if final_sigmas_type not in ("sigma_min", "zero"):
            raise ValueError(f"final_sigmas_type must be 'sigma_min' or 'zero', got {final_sigmas_type!r}")
        self.final_sigmas_type = final_sigmas_type

    def plan(self, start=0):
        n = self.n
        ts = [int(round(v)) for v in np.linspace(0, self.n_train - 1, n + 1)[1:][::-1]]
        alpha = np.sqrt(self.abar)
        sigma = np.sqrt(1.0 - self.abar)
        lam = np.log(alpha) - np.log(sigma)
        out = []
        lower_order_stepped = 0
        for i, t in enumerate(ts):
            if i < start:
                continue
            p = ts[i + 1] if i + 1 < n else 0
            lower_final = (i == n - 1) and n < 15
            lower_second = (i == n - 2) and n < 15
            first = lower_order_stepped < 1 or lower_final or lower_second
            x0_cx = 1.0 / alpha[t]
            x0_ce = -sigma[t] / alpha[t]
            h = lam[p] - lam[t]
            A = -alpha[p] * (math.exp(-h) - 1.0)
            ch = [0.0] * 4
            slot, prev_slot = i % 2, (i - 1) % 2
            if i == n - 1 and self.final_sigmas_type == "zero":
                cx, ce, n_hist = x0_cx, x0_ce, 0      # sigma_next = 0, alpha_next = 1: x_prev = x0 (first order)
            elif first:
                cx = sigma[p] / sigma[t] + A * x0_cx
                ce = A * x0_ce
                n_hist = 0
            else:
                h0 = lam[t] - lam[ts[i - 1]]
                r0 = h0 / h
                c0 = A * (1.0 + 0.5 / r0)
                cx = sigma[p] / sigma[t] + c0 * x0_cx
                ce = c0 * x0_ce
                ch[prev_slot] = -0.5 * A / r0
                n_hist = 2
            out.append(StepPlan(t, cx, ce, ch, x0_cx, x0_ce, [0.0] * 4, n_hist=n_hist, push_x0_slot=slot))
            if lower_order_stepped < 2:
                lower_order_stepped += 1
        return out


class PNDMScheduler(_Base):
    """PLMS (skip_prk_steps) epsilon prediction (Scheduler.swift:137-344): num_steps + 1 UNet calls
    (the second timestep is visited twice).  History ring: eps in slots 0..2, the saved first
    sample (`currentSample`) in slot 3."""

    def __init__(self, num_inference_steps, steps_offset=1, **kw):
        super().__init__(num_inference_steps, **kw)
        self.steps_offset = steps_offset

    def _prev_coeffs(self, t, tp):
        a_t = self.abar[t]
        a_p = self.abar[max(0, tp)]
        b_t, b_p = 1 - a_t, 1 - a_p
        sample_coeff = math.sqrt(a_p / a_t)
        denom = a_t * math.sqrt(b_p) + math.sqrt(a_t * b_t * a_p)
        return sample_coeff, -(a_p - a_t) / denom

    def plan(self, start=0):
        ratio = self.n_train // self.n
        fwd = [int(round(i * float(ratio))) + self.steps_offset for i in range(self.n)]
        ts = fwd[:-1]
        ts = ts + [ts[-1]] if ts else []
        ts = (ts + [fwd[-1]])[::-1]
        # image-to-image: the Swift pipeline slices this list (timeSteps[startStep...], Scheduler.swift:109-114) and
        # feeds it to a fresh scheduler, whose counter-driven branches then apply to whatever comes first
        ts = ts[start:]
        alpha = np.sqrt(self.abar)
        sigma = np.sqrt(1.0 - self.abar)
        out = []
        n_ets = 0  # eps pushed so far
        for counter, t_unet in enumerate(ts):
            t, tp = t_unet, t_unet - ratio
            ch = [0.0] * 4
            x0_ch = [0.0] * 4
            push_eps, push_x = -1, -1
            if counter != 1:
                push_eps = n_ets % 3
                n_ets += 1
                k = min(n_ets, 4)  # entries of `ets` available including the current eps
            else:
                tp, t = t, t + ratio
                k = 0
            sc, mc = self._prev_coeffs(t, tp)
            slot_back = lambda b: (n_ets - b) % 3  # ets[back: b], b >= 2 (b == 1 is the current eps)
            if counter == 0:
                w_cur, w_hist, use_saved = 1.0, {}, False
                push_x = 3
            elif counter == 1:
                w_cur, w_hist, use_saved = 0.5, {(n_ets - 1) % 3: 0.5}, True
            elif k == 2:
                w_cur, w_hist, use_saved = 1.5, {slot_back(2): -0.5}, False
            elif k == 3:
                w_cur, w_hist, use_saved = 23 / 12, {slot_back(2): -16 / 12, slot_back(3): 5 / 12}, False
            else:
                w_cur = 55 / 24
                w_hist = {slot_back(2): -59 / 24, slot_back(3): 37 / 24, slot_back(4): -9 / 24}
                use_saved = False
            # x_prev = sc * sample + mc * e ; x0 = (sample - sigma_t e) / alpha_t ; e = w_cur eps + sum w h
            a_t, s_t = alpha[t], sigma[t]
            cx = 0.0 if use_saved else sc
            x0_cx = 0.0 if use_saved else 1.0 / a_t
            if use_saved:
                ch[3] += sc
                x0_ch[3] += 1.0 / a_t
            ce = mc * w_cur
            x0_ce = -s_t / a_t * w_cur
            for s, wv in w_hist.items():
                ch[s] += mc * wv
                x0_ch[s] += -s_t / a_t * wv
            n_hist = 4 if (use_saved or w_hist) else 0
            out.append(StepPlan(t_unet, cx, ce, ch, x0_cx, x0_ce, x0_ch, n_hist=n_hist, push_eps_slot=push_eps,
                                push_x_slot=push_x))
        return out


class _SigmaBase(_Base):
    """Shared schedule of the sigma-space samplers (diffusers 0.30.2 ``EulerDiscreteScheduler.set_timesteps``, also
    used by the ancestral and LMS schedulers): ``sigma(t) = sqrt((1 - abar_t) / abar_t)`` interpolated at (possibly
    non-integer) timesteps, a final sigma of 0 appended.  The sample lives in sigma space (``x = x_ddim / sqrt(abar_t)``);
    the UNet sees ``x / sqrt(sigma^2 + 1)`` and the timestep ``float(np.float16(t))`` (pipeline.py:504-511).

    ``timestep_spacing``: ``"linspace"`` (the default; what ``from_config`` yields for SD-1.x / 2.x configs, which have
    no such key), ``"leading"`` (SDXL configs, with ``steps_offset``) or ``"trailing"``."""

    SPACINGS = ("linspace", "leading", "trailing")

    def __init__(self, num_inference_steps, timestep_spacing="linspace", steps_offset=1, **kw):
        super().__init__(num_inference_steps, **kw)
        if timestep_spacing not in self.SPACINGS:
            raise ValueError(f"timestep_spacing must be one of {self.SPACINGS}, got {timestep_spacing!r}")
        self.timestep_spacing = timestep_spacing
        self.steps_offset = int(steps_offset)
        n, n_train = self.n, self.n_train
        if timestep_spacing == "linspace":
            ts = np.linspace(0, n_train - 1, n, dtype=np.float32)[::-1].copy()
        elif timestep_spacing == "leading":
            ratio = n_train // n
            ts = (np.arange(0, n) * ratio).round()[::-1].copy().astype(np.float32)
            ts += np.float32(self.steps_offset)
        else:
            ratio = n_train / n
            ts = np.arange(n_train, 0, -ratio).round().copy().astype(np.float32)
            ts -= np.float32(1)
        train_sigmas = np.sqrt((1.0 - self.abar) / self.abar)
        self.raw_timesteps = ts
        self.sigmas = np.concatenate([np.interp(ts.astype(np.float64), np.arange(n_train), train_sigmas), [0.0]])
        smax = float(self.sigmas.max())
        self.init_noise_sigma = smax if timestep_spacing in ("linspace", "trailing") else math.sqrt(smax * smax + 1.0)

    @staticmethod
    def c_in(sigma):
        return 1.0 / math.sqrt(sigma * sigma + 1.0)

    def scale_model_input(self, x, step_index):
        return x * np.float32(self.c_in(self.sigmas[step_index]))

    def first_in_scale(self, start=0):
        return self.c_in(self.sigmas[start])

    def add_noise(self, original_sample, noise, strength):
        """x0 + sigma * noise at the start step (diffusers ``add_noise`` of the sigma schedulers)."""
        s = np.float32(self.sigmas[self.start_step(strength)])
        return original_sample + s * noise

    def _step(self, i, j):
        """Plan of absolute step ``i``, the ``j``-th step since the loop started (multistep state empty at j = 0)."""
        raise NotImplementedError

    def plan(self, start=0):
        out = []
        for j, i in enumerate(range(start, self.n)):
            st = self._step(i, j)
            st.timestep = float(np.float16(self.raw_timesteps[i]))
            st.in_scale = self.c_in(self.sigmas[i + 1])
            out.append(st)
        return out


class EulerDiscreteScheduler(_SigmaBase):
    """diffusers 0.30.2 ``EulerDiscreteScheduler`` (epsilon prediction, s_churn = 0): ``x0 = x - sigma * eps``,
    ``x_prev = x + (sigma_next - sigma) * eps``."""

    def _step(self, i, j):
        s, sn = self.sigmas[i], self.sigmas[i + 1]
        return StepPlan(0.0, 1.0, sn - s, [0.0] * 4, 1.0, -s, [0.0] * 4)


class EulerAncestralDiscreteScheduler(_SigmaBase):
    """diffusers 0.30.2 ``EulerAncestralDiscreteScheduler`` (epsilon prediction): ``sigma_up = sqrt(sigma_next^2 *
    (sigma^2 - sigma_next^2) / sigma^2)``, ``sigma_down = sqrt(sigma_next^2 - sigma_up^2)``,
    ``x_prev = x + (sigma_down - sigma) * eps + sigma_up * z``."""

    @property
    def uses_noise(self):
        return True

    def _step(self, i, j):
        s, sn = self.sigmas[i], self.sigmas[i + 1]
        up = math.sqrt(sn * sn * (s * s - sn * sn) / (s * s))
        down = math.sqrt(max(sn * sn - up * up, 0.0))
        return StepPlan(0.0, 1.0, down - s, [0.0] * 4, 1.0, -s, [0.0] * 4, noise_scale=up, noise_draw=1 + j)


def lms_coefficients(sigmas, i, order):
    """c_k = integral from sigma_i to sigma_{i+1} of the Lagrange basis polynomial of node sigma_{i-k} over the nodes
    sigma_i .. sigma_{i-order+1}, k = 0 .. order-1, in closed form (numpy.polynomial, float64).  The polynomials are
    written in tau - sigma_i, so the integral is one evaluation at sigma_{i+1} - sigma_i without cancellation."""
    from numpy.polynomial import polynomial as P
    base = sigmas[i]
    nodes = [sigmas[i - m] - base for m in range(order)]
    out = []
    for k in range(order):
        p = np.array([1.0])
        for m in range(order):
            if m != k:
                p = P.polymul(p, [-nodes[m], 1.0]) / (nodes[k] - nodes[m])
        out.append(float(P.polyval(sigmas[i + 1] - base, P.polyint(p))))
    return out


class LMSDiscreteScheduler(_SigmaBase):
    """diffusers 0.30.2 ``LMSDiscreteScheduler`` (order 4, epsilon prediction): ``x_prev = x + sum_k c_k eps_{i-k}``,
    ``order = min(steps so far + 1, 4)``, ``c_k`` from ``lms_coefficients``.  The derivative ``(x - x0) / sigma`` is
    ``eps`` itself, so the history ring holds past eps: step ``j`` since the start pushes to slot ``j % 3``."""
    order = 4

    def _step(self, i, j):
        order = min(j + 1, self.order)
        c = lms_coefficients(self.sigmas, i, order)
        ch = [0.0] * 4
        for k in range(1, order):
            ch[(j - k) % 3] = c[k]
        return StepPlan(0.0, 1.0, c[0], ch, 1.0, -self.sigmas[i], [0.0] * 4, n_hist=3 if order > 1 else 0,
                        push_eps_slot=j % 3)


SCHEDULER_MAP = {
    "DDIM": DDIMScheduler,
    "DPMSolverMultistep": DPMSolverMultistepScheduler,
    "EulerAncestralDiscrete": EulerAncestralDiscreteScheduler,
    "EulerDiscrete": EulerDiscreteScheduler,
    "LMSDiscrete": LMSDiscreteScheduler,
    "PNDM": PNDMScheduler,
}


def make_scheduler(name, num_inference_steps, **kw):
    if name not in SCHEDULER_MAP:
        raise ValueError(f"unsupported scheduler {name!r}; available: {sorted(SCHEDULER_MAP)}")
    return SCHEDULER_MAP[name](num_inference_steps, **kw)


def apply_plan_host(step: StepPlan, guidance, eps_uncond, eps_text, x, hist, noise=None, return_unet_in=False):
    """numpy mirror of the device kernel's arithmetic (host-logic tests only).  ``noise``: the step's normals (needed
    when ``step.noise_scale != 0``); ``return_unet_in``: also return the next UNet input ``in_scale * x_prev``."""
    eps = eps_uncond + guidance * (eps_text - eps_uncond)
    xp = step.cx * x + step.ce * eps
    x0 = step.x0_cx * x + step.x0_ce * eps
    for j in range(step.n_hist):
        xp = xp + step.ch[j] * hist[j]
        x0 = x0 + step.x0_ch[j] * hist[j]
    if step.noise_scale != 0.0:
        if noise is None:
            raise ValueError("this step adds noise: pass `noise`")
        xp = xp + step.noise_scale * noise
    if step.push_eps_slot >= 0:
        hist[step.push_eps_slot] = eps
    if step.push_x0_slot >= 0:
        hist[step.push_x0_slot] = x0
    if step.push_x_slot >= 0:
        hist[step.push_x_slot] = x
    if return_unet_in:
        return xp, x0, step.in_scale * xp
    return xp, x0
