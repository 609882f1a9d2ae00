"""Text-to-image pipeline with the reference's call surface, running on the B200 kernels.

Mirrors ``CoreMLStableDiffusionPipeline.__call__`` (``python_coreml_stable_diffusion/pipeline.py:403-589``):
same keyword arguments, same order of operations (encode -> latents -> [CFG-duplicated UNet ->
guidance -> scheduler.step] x N -> VAE decode -> clip -> NHWC -> PIL), same
``StableDiffusionPipelineOutput(images, nsfw_content_detected)`` result.  Differences, all by design:

* the loop body stays on the GPU: UNet (CUDA graph), then ONE fused kernel for guidance + scheduler
  step; there is no per-step host round trip (the reference crosses numpy<->Core ML twice per step);
* batches of prompts are accepted (the reference raises ``NotImplementedError``, pipeline.py:434-438;
  BASELINE config 3 needs 8 prompts per GPU);
* the CLIP text encoder / tokenizer are not part of this round's hot path (SURVEY 8f N2): prompts
  are turned into *synthetic* 77-token embeddings by ``SyntheticTextEncoder`` unless the caller
  passes ``prompt_embeds`` or installs a real ``text_encoder`` callable with the reference contract
  (``input_ids`` float32 (1, 77) -> ``last_hidden_state`` (1, 77, D), pipeline.py:151-175).
"""
from __future__ import annotations

import dataclasses
import hashlib
from typing import List, Optional, Tuple, Union

import numpy as np
import torch

from . import config as C
from . import lib as L
from . import scheduler as S
from .model import UNetModel
from .vae import VAEDecoderModel


@dataclasses.dataclass
class StableDiffusionPipelineOutput:
    images: Union[List, np.ndarray]
    nsfw_content_detected: Optional[List[bool]]


class SyntheticTokenizer:
    """Deterministic stand-in for the CLIP BPE tokenizer: whitespace words -> ids by hash, padded to
    ``model_max_length`` with the end-of-text id (same padding convention as pipeline.py:151-158)."""
    model_max_length = 77
    bos, eos, vocab = 49406, 49407, 49408

    def __call__(self, text: str):
        ids = [self.bos]
        for wd in text.lower().split()[: self.model_max_length - 2]:
            ids.append(int.from_bytes(hashlib.sha256(wd.encode()).digest()[:4], "little") % (self.bos - 1) + 1)
        ids.append(self.eos)
        ids += [self.eos] * (self.model_max_length - len(ids))
        return np.array([ids], dtype=np.float32)  # the reference feeds input_ids as float32 (pipeline.py:173)


class SyntheticTextEncoder:
    """Maps token ids to fixed pseudo-random unit-variance embeddings (no weights exist offline)."""

    def __init__(self, hidden=1024, seq=77):
        self.hidden, self.seq = hidden, seq
        self.expected_inputs = {"input_ids": {"shape": (1, seq), "dtype": np.dtype(np.float32)}}

    def __call__(self, input_ids):
        out = np.empty((1, self.seq, self.hidden), dtype=np.float32)
        for i, tok in enumerate(np.asarray(input_ids).reshape(-1).astype(np.int64)):
            out[0, i] = np.random.RandomState(int(tok) * 131 + i).standard_normal(self.hidden)
        return {"last_hidden_state": out}


class B200StableDiffusionPipeline:
    """Drop-in for ``CoreMLStableDiffusionPipeline`` on one B200."""

    def __init__(self, unet: UNetModel, vae_decoder: VAEDecoderModel, scheduler="DDIM", text_encoder=None,
                 tokenizer=None, force_zeros_for_empty_prompt=True, xl=False, controlnet=None, loop_graph=True,
                 vae_encoder=None, text_encoder_2=None, tokenizer_2=None, scheduler_kwargs=None, unet_refiner=None):
        self.unet = unet
        # SDXL refiner UNet (StableDiffusionXLPipeline.swift:205-225): takes over the loop at step
        # int(len(timesteps) * refiner_start) with its own conditioning (set_refiner_inputs)
        self.unet_refiner = unet_refiner
        self.text_encoder_2 = text_encoder_2  # SDXL: CLIPTextModelWithProjection slot (pipeline.py:64-65, 136-141)
        self.tokenizer_2 = tokenizer_2
        self.vae_encoder = vae_encoder  # VAEEncoderModel or None (image-to-image, StableDiffusionPipeline.swift:371-376)
        self.loop_graph = bool(loop_graph) and unet.use_cuda_graph  # whole-loop CUDA graph (denoise())
        self._loop_graphs = {}
        self.controlnet = list(controlnet) if controlnet else None  # pipeline.py:66,106: Optional[List[model]]
        if self.controlnet and not unet.engine.support_controlnet:
            raise ValueError("the UNet was not built with support_controlnet=True (no additional_residual inputs)")
        self.vae_decoder = vae_decoder
        self.scheduler_name = scheduler
        # this class mirrors the reference's PYTHON pipeline, whose DPM-Solver++ is diffusers 0.30.2
        # (final_sigmas_type="zero"); pass scheduler_kwargs={"final_sigmas_type": "sigma_min"} for the Swift CLI's ending
        self.scheduler_kwargs = dict(scheduler_kwargs or {})
        if scheduler == "DPMSolverMultistep":
            self.scheduler_kwargs.setdefault("final_sigmas_type", "zero")
        self.device = unet.device
        self.xl = xl
        d_ctx = unet.engine.cfg["cross_attention_dim"]
        self.text_encoder = text_encoder or SyntheticTextEncoder(d_ctx, unet.seq)
        self.tokenizer = tokenizer or SyntheticTokenizer()
        self.force_zeros_for_empty_prompt = force_zeros_for_empty_prompt
        self.vae_scale_factor = vae_decoder.scale
        self.height = unet.h * self.vae_scale_factor
        self.width = unet.w * self.vae_scale_factor
        self.images_per_call = unet.batch // 2
        n, c, h, w = self.images_per_call, unet.in_channels, unet.h, unet.w
        dev = self.device
        self._latents = torch.zeros(n, c, h, w, dtype=torch.float32, device=dev)
        self._hist = torch.zeros(4, n, c, h, w, dtype=torch.float32, device=dev)
        self._denoised = torch.zeros(n, c, h, w, dtype=torch.float32, device=dev)
        self._ctx = torch.zeros(2 * n, d_ctx, 1, unet.seq, dtype=torch.float16, device=dev)
        self._t = torch.zeros(2 * n, dtype=torch.float32, device=dev)
        # Philox key of the samplers' per-step noise (b200sd_sampler_step): device memory, so a new seed is a copy, not a
        # new loop graph
        self._rng_key = torch.zeros(2, dtype=torch.int32, device=dev)

    # ---------------------------------------------------------------- factory
    @classmethod
    def from_random_init(cls, model_version="sd21-base", images_per_call=1, device="cuda", seed=0,
                         scheduler="DDIM", height=512, width=512, unet_cfg=None, vae_cfg=None, controlnet_cfgs=None,
                         text_encoder_cfg=None, tokenizer=None, with_vae_encoder=False):
        """Random-init weights of the named architecture (no checkpoints exist offline).  ``controlnet_cfgs``:
        list of ControlNet configs (seeded seed+2, seed+3, ...); switches the UNet to its control variant.
        ``text_encoder_cfg``: a CLIP text config (config.OPENCLIP_H_TEXT for SD-2.x) -> the text encoder runs on the
        device (random-init, seed+100) instead of the synthetic embedding table; ``tokenizer``: e.g. a
        ``tokenizer.BPETokenizer`` built from the checkpoint's vocab.json / merges.txt."""
        unet_cfg = unet_cfg or {"sd21-base": C.SD21_BASE_UNET, "sdxl-base": C.SDXL_BASE_UNET,
                                "tiny": C.TINY_UNET}[model_version]
        vae_cfg = vae_cfg or (C.TINY_VAE if model_version == "tiny" else C.SD_VAE)
        if controlnet_cfgs:
            unet_cfg = dict(unet_cfg, support_controlnet=True)
        f = 2 ** (len(vae_cfg["block_out_channels"]) - 1)
        usd = C.random_state_dict(C.unet_param_shapes(unet_cfg), seed=seed, dtype=torch.float16)
        vsd = C.random_state_dict(C.vae_decoder_param_shapes(vae_cfg), seed=seed + 1, dtype=torch.float16)
        unet = UNetModel(unet_cfg, usd, batch=2 * images_per_call, height=height // f, width=width // f,
                         device=device)
        vae = VAEDecoderModel(vae_cfg, vsd, batch=images_per_call, height=height // f, width=width // f,
                              device=device)
        nets = None
        if controlnet_cfgs:
            from .controlnet import ControlNetModel
            nets = [ControlNetModel(c, C.random_state_dict(C.controlnet_param_shapes(c), seed=seed + 2 + i,
                                                           dtype=torch.float16),
                                    batch=2 * images_per_call, height=height // f, width=width // f, device=device)
                    for i, c in enumerate(controlnet_cfgs)]
        enc = None
        if text_encoder_cfg is not None:
            from .text_encoder import TextEncoderModel
            if text_encoder_cfg["hidden_size"] != unet_cfg["cross_attention_dim"]:
                raise ValueError("text encoder width does not match the UNet's cross_attention_dim")
            enc = TextEncoderModel(text_encoder_cfg, C.random_clip_text_state_dict(text_encoder_cfg, seed=seed + 100,
                                                                                   dtype=torch.float16),
                                   batch=1, device=device)
        venc = None
        if with_vae_encoder:
            from .vae import VAEEncoderModel
            esd = C.random_state_dict(C.vae_encoder_param_shapes(vae_cfg), seed=seed + 50, dtype=torch.float16)
            venc = VAEEncoderModel(vae_cfg, esd, batch=images_per_call, height=height, width=width, device=device)
        return cls(unet, vae, scheduler=scheduler, xl=unet.engine.xl, controlnet=nets, text_encoder=enc,
                   tokenizer=tokenizer, vae_encoder=venc, force_zeros_for_empty_prompt=unet.engine.xl)

    _SCHEDULER_CLASS = {"PNDMScheduler": "PNDM", "DDIMScheduler": "DDIM", "DPMSolverMultistepScheduler": "DPMSolverMultistep"}
    _SIGMA_SCHEDULERS = ("EulerDiscrete", "EulerAncestralDiscrete", "LMSDiscrete")

    @classmethod
    def from_pretrained(cls, model_dir, images_per_call=1, device="cuda", height=None, width=None,
                        scheduler_override=None, controlnet_dirs=None, force_zeros_for_empty_prompt=None,
                        with_vae_encoder=False, refiner_dir=None):
        """Build the pipeline from a diffusers-layout model directory (``unet/``, ``vae/``, ``text_encoder[_2]/``,
        ``tokenizer[_2]/``, ``scheduler/``): the counterpart of ``get_coreml_pipe(pytorch_pipe, mlpackages_dir,
        model_version, compute_unit, scheduler_override, controlnet_models, force_zeros_for_empty_prompt)``
        (pipeline.py:607-697), which wires converted .mlpackage files to the same slots.  Weights are read with
        ``checkpoint.load_component`` (schema-checked), configs with ``checkpoint.read_config``.
        ``refiner_dir``: an SDXL refiner directory whose UNet takes over at ``refiner_start`` (``__call__``)."""
        import json
        import os
        from . import checkpoint as K
        from .text_encoder import TextEncoderModel
        from .tokenizer import BPETokenizer

        ucfg = K.read_config(model_dir, "unet")
        vcfg = K.read_config(model_dir, "vae")
        if controlnet_dirs:
            ucfg = dict(ucfg, support_controlnet=True)
        f = 2 ** (len(vcfg["block_out_channels"]) - 1)
        size = ucfg.get("sample_size", 64)
        h = (height // f) if height else size
        w = (width // f) if width else size
        xl = ucfg.get("addition_embed_type") == "text_time"
        unet = UNetModel(ucfg, K.load_component(model_dir, "unet", ucfg), batch=2 * images_per_call, height=h, width=w,
                         device=device)
        vsd = K.read_state_dict(os.path.join(model_dir, "vae"))
        vae = VAEDecoderModel(vcfg, K.check_state_dict("vae_decoder", vcfg, vsd), batch=images_per_call, height=h,
                              width=w, device=device)
        venc = None
        if with_vae_encoder:
            from .vae import VAEEncoderModel
            venc = VAEEncoderModel(vcfg, K.check_state_dict("vae_encoder", vcfg, vsd), batch=images_per_call,
                                   height=h * f, width=w * f, device=device)

        def text_pair(enc_dir, tok_dir):
            if not os.path.isdir(os.path.join(model_dir, enc_dir)):
                return None, None
            tcfg = K.read_config(model_dir, enc_dir)
            # SDXL conditions on hidden_states[-2] of both encoders (torch2coreml.py:416-446: ``hidden_embeds``)
            enc = TextEncoderModel(tcfg, K.load_component(model_dir, enc_dir, tcfg), batch=1, device=device,
                                   hidden_layer=-2 if xl else None)
            tok = None
            tdir = os.path.join(model_dir, tok_dir)
            if os.path.exists(os.path.join(tdir, "merges.txt")):
                pad = "<|endoftext|>"
                stm = os.path.join(tdir, "special_tokens_map.json")  # SDXL's second tokenizer pads with "!"
                if os.path.exists(stm):
                    with open(stm) as fh:
                        pt = json.load(fh).get("pad_token", pad)
                    pad = pt.get("content", pad) if isinstance(pt, dict) else pt
                tok = BPETokenizer.from_files(os.path.join(tdir, "merges.txt"), os.path.join(tdir, "vocab.json"), pad_token=pad)
            return enc, tok

        enc1, tok1 = text_pair("text_encoder", "tokenizer")
        enc2, tok2 = text_pair("text_encoder_2", "tokenizer_2")
        sched = scheduler_override
        sched_cfg_path = os.path.join(model_dir, "scheduler", "scheduler_config.json")
        sched_cfg = {}
        if sched is None or os.path.exists(sched_cfg_path):  # without an override the config must exist
            with open(sched_cfg_path) as fh:
                sched_cfg = json.load(fh)
        sched_kwargs = None
        if sched in cls._SIGMA_SCHEDULERS:
            # what the reference's from_config carries over to these classes (pipeline.py:816-821)
            sched_kwargs = {k: sched_cfg[k] for k in ("timestep_spacing", "steps_offset") if k in sched_cfg}
        if sched is None:
            name = sched_cfg.get("_class_name", "PNDMScheduler")
            if name not in cls._SCHEDULER_CLASS:
                raise ValueError(f"scheduler {name} of the checkpoint is not implemented; pass scheduler_override "
                                 f"(one of {sorted(S.SCHEDULER_MAP)})")
            sched = cls._SCHEDULER_CLASS[name]
        nets = None
        if controlnet_dirs:
            from .controlnet import ControlNetModel
            nets = []
            for d in controlnet_dirs:
                with open(os.path.join(d, "config.json")) as fh:
                    ccfg = {k: (tuple(v) if isinstance(v, list) else v) for k, v in json.load(fh).items() if not k.startswith("_")}
                nets.append(ControlNetModel(ccfg, K.load_component(d, "controlnet", ccfg), batch=2 * images_per_call,
                                            height=h, width=w, device=device))
        refiner = None
        if refiner_dir:
            rcfg = K.read_config(refiner_dir, "unet")
            refiner = UNetModel(rcfg, K.load_component(refiner_dir, "unet", rcfg), batch=2 * images_per_call, height=h,
                                width=w, device=device)
        if force_zeros_for_empty_prompt is None:
            force_zeros_for_empty_prompt = xl   # the reference's CLI sets it for SDXL only (pipeline.py:744-755)
        return cls(unet, vae, scheduler=sched, text_encoder=enc1, tokenizer=tok1, text_encoder_2=enc2, tokenizer_2=tok2,
                   xl=xl, controlnet=nets, vae_encoder=venc, force_zeros_for_empty_prompt=force_zeros_for_empty_prompt,
                   unet_refiner=refiner, scheduler_kwargs=sched_kwargs)

    # ---------------------------------------------------------------- reference-named helpers
    def check_inputs(self, prompt, height, width, callback_steps):
        """pipeline.py:359-382."""
        if not isinstance(prompt, (str, list)):
            raise ValueError(f"`prompt` has to be of type `str` or `list` but is {type(prompt)}")
        if height % 8 != 0 or width % 8 != 0:
            raise ValueError(f"`height` and `width` have to be divisible by 8 but are {height} and {width}.")
        if callback_steps is None or not isinstance(callback_steps, int) or callback_steps <= 0:
            raise ValueError(f"`callback_steps` has to be a positive integer but is {callback_steps} of type "
                             f"{type(callback_steps)}.")

    def _encode_one(self, text):
        ids = self.tokenizer(text)
        return np.asarray(self.text_encoder(input_ids=ids)["last_hidden_state"], dtype=np.float32)[0]  # (S, D)

    def _encode_prompt(self, prompts, do_cfg, negative_prompt):
        """-> (2B, D, 1, S) fp16 array, uncond half first (pipeline.py:123-257: concat [neg, pos], :252 transpose)."""
        conds = [self._encode_one(p) for p in prompts]
        if isinstance(negative_prompt, list):
            if len(negative_prompt) != len(prompts):
                raise ValueError(f"`negative_prompt` has batch size {len(negative_prompt)}, but `prompt` has batch size "
                                 f"{len(prompts)}")
            negs = list(negative_prompt)
        else:
            negs = [negative_prompt] * len(prompts)
        unconds = []
        for ng, cnd in zip(negs, conds):
            if not do_cfg:
                unconds.append(cnd)
            elif ng is None and self.force_zeros_for_empty_prompt:
                # pipeline.py:183-184: zeros only when NO negative prompt was given and the flag is set (the
                # reference's CLI sets it for SDXL only, pipeline.py:744-755); an explicit "" is encoded
                unconds.append(np.zeros_like(cnd))
            else:
                unconds.append(self._encode_one(ng or ""))
        emb = np.stack(unconds + conds, 0)  # (2B, S, D)
        return np.ascontiguousarray(emb.transpose(0, 2, 1)[:, :, None, :]).astype(np.float16)

    def _encode_prompt_xl(self, prompts, do_cfg, negative_prompt=None, prompts_2=None, negative_prompt_2=None,
                          only_second=False):
        """SDXL branch of pipeline.py:123-257: both encoders' ``hidden_embeds`` concatenated along the feature axis
        (encoder 1 first), the pooled output of the LAST encoder, zeros for the negative branch when no negative
        prompt is given and force_zeros_for_empty_prompt.  The refiner has only encoder 2 (text_encoder is None).
        -> ((2B, D1 + D2, 1, S) fp16, (2B, P) fp32), uncond half first."""
        pairs = [(self.tokenizer, self.text_encoder), (self.tokenizer_2, self.text_encoder_2)]
        if self.text_encoder is None or only_second:  # the refiner is conditioned on the second encoder only
            pairs = pairs[1:]
        texts = [prompts, prompts_2 if prompts_2 is not None else prompts][-len(pairs):]

        def run(text_lists):
            per_prompt, pooled = [], []
            for i in range(len(text_lists[0])):
                feats = []
                for (tok, enc), tl in zip(pairs, text_lists):
                    o = enc(input_ids=np.asarray(tok(tl[i]), dtype=np.float32))
                    feats.append(np.asarray(o["hidden_embeds"], dtype=np.float32)[0])
                    last_pooled = np.asarray(o["pooled_outputs"], dtype=np.float32)[0]
                per_prompt.append(np.concatenate(feats, axis=-1))  # (S, D1 + D2)
                pooled.append(last_pooled)
            return np.stack(per_prompt, 0), np.stack(pooled, 0)

        emb, pooled = run(texts)
        if do_cfg:
            if negative_prompt is None and self.force_zeros_for_empty_prompt:
                neg, neg_pooled = np.zeros_like(emb), np.zeros_like(pooled)
            else:
                neg_1 = negative_prompt or ""
                neg_2 = negative_prompt_2 or neg_1
                as_list = lambda v: [v] * len(prompts) if isinstance(v, str) else list(v)  # noqa: E731
                neg_1, neg_2 = as_list(neg_1), as_list(neg_2)
                if len(neg_1) != len(prompts):
                    raise ValueError(f"`negative_prompt` has batch size {len(neg_1)}, but `prompt` has batch size "
                                     f"{len(prompts)}")
                neg, neg_pooled = run([neg_1, neg_2][-len(pairs):])
            emb, pooled = np.concatenate([neg, emb], 0), np.concatenate([neg_pooled, pooled], 0)
        else:
            # the UNet always runs both batch halves: without guidance both carry the prompt (like _encode_prompt)
            emb, pooled = np.concatenate([emb, emb], 0), np.concatenate([pooled, pooled], 0)
        return np.ascontiguousarray(emb.transpose(0, 2, 1)[:, :, None, :]).astype(np.float16), pooled

    def prepare_latents(self, batch, channels, height, width, latents=None, seed=None, rng="numpy"):
        """pipeline.py:322-344: np.random.randn(...).astype(fp16) * init_noise_sigma (the global numpy stream, seeded by
        the caller like pipeline.py:725-726).  With ``seed``: the Swift pipeline's ``generateLatentSamples``
        (StableDiffusionPipeline.swift:361-379): one draw of C*h*w normals per image from the chosen
        ``StableDiffusionRNG`` source (numpy / torch / nvidia, rng.py), so a seed reproduces the reference CLIs' latents."""
        shape = (batch, channels, height // self.vae_scale_factor, width // self.vae_scale_factor)
        if latents is None and seed is not None:
            from .rng import random_source
            src = random_source(rng, seed)
            per = int(np.prod(shape[1:]))
            latents = np.stack([src.normal_array(per).reshape(shape[1:]) for _ in range(batch)]).astype(np.float32)
        elif latents is None:
            latents = np.random.randn(*shape).astype(np.float16)
        elif tuple(latents.shape) != shape:
            raise ValueError(f"Unexpected latents shape, got {latents.shape}, expected {shape}")
        return latents.astype(np.float32) * 1.0

    def prepare_control_cond(self, controlnet_cond, do_classifier_free_guidance, batch_size, num_images_per_prompt):
        """pipeline.py:345-356: each (3, H, W) condition image is repeated per image and doubled for CFG."""
        out = []
        for cond in controlnet_cond:
            cond = np.stack([np.asarray(cond)] * batch_size * num_images_per_prompt)
            # doubled like the latents: this engine always runs both batch halves (with guidance <= 1 both carry the
            # prompt), where the reference doubles only under guidance (pipeline.py:345-356)
            cond = np.concatenate([cond] * 2)
            out.append(cond)
        return out

    def run_controlnet(self, sample, timestep, encoder_hidden_states, controlnet_cond):
        """pipeline.py:259-284 on the device: every ControlNet sees the same UNet inputs; their residuals are
        summed (fp16, like the reference's in-place numpy add).  Returns NCHW views of NHWC fp16 tensors."""
        if not self.controlnet:
            raise ValueError("Conditions for controlnet are given but the pipeline has no controlnet modules")
        total = None
        for module, cond in zip(self.controlnet, controlnet_cond):
            module._sample.copy_(sample)
            module._t.copy_(timestep)
            module._ctx.copy_(encoder_hidden_states)
            module._cond.copy_(cond)
            outs = module.forward_device()
            if total is None:
                total = list(outs)
            else:
                for acc, o in zip(total, outs):
                    L.add(acc, o, out=acc)
        return [r.permute(0, 3, 1, 2) for r in total]

    @staticmethod
    def numpy_to_pil(images):
        from PIL import Image
        images = (images * 255).round().astype("uint8")
        return [Image.fromarray(im) for im in images]

    # ---------------------------------------------------------------- device loop
    @staticmethod
    def _coeffs(st, guidance_scale, k=None):
        k = k or L.StepCoeffs()
        k.guidance = float(guidance_scale)
        k.cx, k.ce, k.x0_cx, k.x0_ce = st.cx, st.ce, st.x0_cx, st.x0_ce
        for j in range(4):
            k.ch[j] = st.ch[j]
            k.x0_ch[j] = st.x0_ch[j]
        k.n_hist, k.push_eps_slot, k.push_x0_slot, k.push_x_slot = (st.n_hist, st.push_eps_slot,
                                                                    st.push_x0_slot, st.push_x_slot)
        return k

    def _sampler_coeffs(self, st, guidance_scale, k=None):
        """b200sd_sampler_coeffs of a step: the linear update + input scale, noise scale and this step's Philox draws."""
        k = k or L.SamplerCoeffs()
        self._coeffs(st, guidance_scale, k.step)
        k.in_scale, k.noise_scale = st.in_scale, st.noise_scale
        k.noise_draw = (self.images_per_call * st.noise_draw) & 0xFFFFFFFF
        return k

    def _make_scheduler(self, num_inference_steps, eta=0.0):
        kw = dict(self.scheduler_kwargs)
        if eta:  # like the reference (pipeline.py:384-396), eta reaches DDIM only and is ignored by the other schedulers
            if self.scheduler_name == "DDIM":
                kw["eta"] = float(eta)
        return S.make_scheduler(self.scheduler_name, num_inference_steps, **kw)

    def _set_noise_key(self, seed):
        """The Philox key of the per-step noise: ``seed``, or with ``seed=None`` a draw from the global numpy stream,
        taken after every other draw of the call."""
        if seed is None:
            seed = int(np.random.randint(0, 2 ** 32, dtype=np.uint64))
        key = np.array([int(seed) & 0xFFFFFFFF, 0], dtype=np.uint32).view(np.int32)
        self._rng_key.copy_(torch.from_numpy(key))

    def _loop_on_static_buffers(self, plan, guidance_scale, ts_rows, use_controlnet=False, refiner_start_step=None,
                                in_scale0=1.0):
        """The whole N-step loop on static device buffers (no host-side tensor arguments): what the loop graph
        captures.  Prologue, once per prompt: cross-attention K/V of all blocks from the text states, the
        time-embedding biases of all ResNet blocks for ALL timesteps (`ts_rows`: each step's timestep repeated per
        batch row, a device tensor made outside the capture), the first UNet input.  Per step: the UNet launch
        sequence and ONE fused kernel for guidance + scheduler update, which also writes the next step's UNet
        input (fp16 NHWC, both CFG halves: pipeline.py:502 np.concatenate([latents] * 2)) -- no fill / copy /
        layout kernels in between."""
        n = self.images_per_call
        rs = len(plan) if refiner_start_step is None else max(0, min(len(plan), refiner_start_step))
        # which UNet runs each step: the SDXL refiner takes over at refiner_start_step with its own conditioning
        # (StableDiffusionXLPipeline.swift:205-225); each model gets its per-prompt prologue and its own time table
        models = [self.unet if i < rs else self.unet_refiner for i in range(len(plan))]
        self._hist.zero_()
        b = self.unet.batch
        tables = {}
        for m, lo, hi in ((self.unet, 0, rs), (self.unet_refiner, rs, len(plan))):
            if hi > lo:
                m.prepare_prompt()
                tables[id(m)] = (m.time_table(ts_rows[lo * b: hi * b]), lo)
        first = models[0]
        L.nchw_to_nhwc(self._latents, c_pad=first.engine.in_pad, out=first._x_nhwc[:n])
        L.nchw_to_nhwc(self._latents, c_pad=first.engine.in_pad, out=first._x_nhwc[n:])
        if in_scale0 != 1.0:  # sigma-space samplers: the UNet sees c_in(sigma_0) * x (pipeline.py:504-508)
            k0 = L.SamplerCoeffs()
            k0.in_scale = in_scale0
            L.sampler_step(None, self._latents, k0, unet_in=first._x_nhwc)
        if use_controlnet:
            self.prepare_controlnets(ts_rows)
        for i, st in enumerate(plan):
            u = models[i]
            table, lo = tables[id(u)]
            u._run_core(table[i - lo], self.controlnet_residuals(i) if use_controlnet else None)
            k = self._sampler_coeffs(st, guidance_scale)
            k.step.noise_pred_nhwc = 1
            nxt = models[i + 1] if i + 1 < len(plan) else u
            L.sampler_step(u._out_nhwc, self._latents, k, hist=self._hist, denoised=self._denoised,
                           unet_in=nxt._x_nhwc, rng_key=self._rng_key)

    def set_control_conditions(self, controlnet_cond):
        """Copy the conditioning images (each (2B, 3, H, W)) into the ControlNets' static input buffers."""
        for module, cond in zip(self.controlnet, controlnet_cond):
            module._cond.copy_(torch.as_tensor(cond))

    def prepare_controlnets(self, ts_rows):
        """Device-loop prologue of every ControlNet: text states, the embedding of its conditioning image (static
        buffer `_cond`), time-embedding table."""
        for module in self.controlnet:
            module._ctx.copy_(self.unet._ctx)
            module.prepare_prompt(ts_rows)

    def controlnet_residuals(self, step, _temb=None):
        """pipeline.py:259-284 inside the device loop: every ControlNet sees the UNet's input; residuals are summed."""
        total = None
        for module in self.controlnet:
            outs = module.run_core(self.unet._x_nhwc, step)
            if total is None:
                total = list(outs)
            else:
                total = [L.add(acc, o) for acc, o in zip(total, outs)]
        return total

    def _ts_rows(self, plan):
        return torch.tensor([float(st.timestep) for st in plan for _ in range(self.unet.batch)], dtype=torch.float32,
                            device=self.device)

    def _loop_graph_for(self, key, plan, guidance_scale, use_controlnet=False, refiner_start_step=None, in_scale0=1.0):
        g = self._loop_graphs.get(key)
        if g is None:
            keep = self._latents.clone()
            ts_rows = self._ts_rows(plan)
            s = torch.cuda.Stream(device=self.device)  # eager warm-up off the capture: workspaces, weight tiling
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self._loop_on_static_buffers(plan[:1], guidance_scale, ts_rows[: self.unet.batch], use_controlnet,
                                             in_scale0=in_scale0)
                if refiner_start_step is not None and refiner_start_step < len(plan):  # warm the refiner's kernels too
                    self._loop_on_static_buffers(plan[-1:], guidance_scale, ts_rows[-self.unet.batch:], use_controlnet, 0,
                                                 in_scale0=in_scale0)
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            self._latents.copy_(keep)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._loop_on_static_buffers(plan, guidance_scale, ts_rows, use_controlnet, refiner_start_step, in_scale0)
            g._b200sd_keep = ts_rows
            self._latents.copy_(keep)  # capture does not execute, but keep the contract obvious
            if len(self._loop_graphs) >= 4:
                self._loop_graphs.pop(next(iter(self._loop_graphs)))
            self._loop_graphs[key] = g
        return g

    def denoise(self, text_embeddings, latents, num_inference_steps, guidance_scale, callback=None,
                callback_steps=1, time_ids=None, text_embeds=None, return_denoised=False, record=None,
                controlnet_cond=None, start_step=0, refiner=None, refiner_start=0.8, eta=0.0, seed=None):
        """Runs the N-step loop (from ``start_step``: image-to-image) entirely on the device.  ``text_embeddings`` (2B, D, 1, S) and ``latents``
        (B, C, h, w) may be numpy (copied once, before the loop) or CUDA tensors.  ``record`` (a list) receives
        (timestep, noise_pred, latents_after_step) clones per step -- a debugging / testing aid.  Without
        callback / record / ControlNet the whole loop replays as ONE CUDA graph (SURVEY 8f N1): the scheduler
        history lives on the device and no host synchronisation happens between the first and the last step.
        ``latents`` are in the scheduler's own space (already multiplied by ``init_noise_sigma``, ``__call__`` does
        that).  ``eta``: DDIM's noise weight.  ``seed``: the Philox key of the per-step noise of Euler-ancestral and
        DDIM eta > 0 (``None``: drawn from the global numpy stream); it is not part of the loop graph."""
        sched = self._make_scheduler(num_inference_steps, eta)
        plan = list(sched.plan(start=start_step)) if start_step else list(sched.plan())
        in_scale0 = sched.first_in_scale(start_step)
        if sched.uses_noise:
            self._set_noise_key(seed)
        n = self.images_per_call
        self._ctx.copy_(torch.as_tensor(text_embeddings), non_blocking=True)
        self._latents.copy_(torch.as_tensor(latents), non_blocking=True)
        if controlnet_cond:
            controlnet_cond = [torch.as_tensor(c).to(self.device, torch.float16) for c in controlnet_cond]
        elif self.unet._res:
            # a UNet built with additional_residual inputs but called without conditions: the static residual buffers
            # would still hold the previous ControlNet call's last step (the reference cannot run this combination)
            for buf in self.unet._res:
                buf.zero_()
        if self.loop_graph and callback is None and record is None:
            u = self.unet
            u._ctx.copy_(self._ctx)
            if u.engine.xl:
                u._time_ids.copy_(torch.as_tensor(time_ids).reshape(u._time_ids.shape))
                u._text_embeds.copy_(torch.as_tensor(text_embeds))
            if controlnet_cond:
                self.set_control_conditions(controlnet_cond)
            rstep = None
            if refiner is not None:
                if self.unet_refiner is None:
                    raise ValueError("refiner inputs were given but the pipeline has no unet_refiner")
                r = self.unet_refiner
                r._ctx.copy_(torch.as_tensor(refiner["encoder_hidden_states"]))
                r._time_ids.copy_(torch.as_tensor(refiner["time_ids"]).reshape(r._time_ids.shape))
                r._text_embeds.copy_(torch.as_tensor(refiner["text_embeds"]))
                rstep = int(np.float32(len(plan)) * np.float32(refiner_start))  # Int(Float(timeSteps.count) * refinerStart)
            key = (self.scheduler_name, int(num_inference_steps), float(guidance_scale), int(start_step),
                   bool(controlnet_cond), tuple(sorted(self.scheduler_kwargs.items())), rstep, float(eta))
            self._loop_graph_for(key, plan, guidance_scale, bool(controlnet_cond), rstep, in_scale0).replay()
            return self._denoised if return_denoised else self._latents
        if refiner is not None:
            raise ValueError("the refiner hand-off runs in the device loop only (no callback / record)")
        self._hist.zero_()
        k = L.SamplerCoeffs()
        scale = in_scale0
        for i, st in enumerate(plan):
            self._t.fill_(float(st.timestep))
            sample = torch.cat([self._latents, self._latents], 0)  # pipeline.py:502
            if scale != 1.0:
                # scale_model_input (pipeline.py:504-508): the fp32 product the step kernel writes to the loop graph's
                # UNet input, rounded to fp16 by the same conversion, so both paths feed the UNet the same bits
                sample.mul_(float(np.float32(scale)))
            residuals = None
            if controlnet_cond:  # pipeline.py:515-529
                residuals = self.run_controlnet(sample, self._t, self._ctx, controlnet_cond)
            noise_pred = self.unet.forward_device(sample, self._t, self._ctx, time_ids, text_embeds, residuals)
            self._sampler_coeffs(st, guidance_scale, k)
            scale = st.in_scale
            if record is not None:
                eps_copy = noise_pred.clone()
            L.sampler_step(noise_pred, self._latents, k, hist=self._hist, denoised=self._denoised, rng_key=self._rng_key)
            if record is not None:
                record.append((st.timestep, eps_copy, self._latents.clone()))
            if callback is not None and i % callback_steps == 0:
                callback(i, st.timestep, self._latents)
        return self._denoised if return_denoised else self._latents

    def decode_latents(self, latents):
        """pipeline.py:313-320 on the device: z / scaling -> decoder -> clip(x/2+0.5, 0, 1) -> NHWC fp32."""
        eng = self.vae_decoder.engine
        self.vae_decoder._z.copy_(latents)
        self.vae_decoder._z.mul_(1.0 / eng.scaling)
        img = eng.forward(self.vae_decoder._z)
        return L.image_postprocess(img, c=eng.out_ch)

    # ---------------------------------------------------------------- public API
    def __call__(self, prompt, height=512, width=512, num_inference_steps=50, guidance_scale=7.5,
                 negative_prompt=None, num_images_per_prompt=1, eta=0.0, latents=None, output_type="pil",
                 return_dict=True, callback=None, callback_steps=1, controlnet_cond=None,
                 original_size: Optional[Tuple[int, int]] = None, crops_coords_top_left: Tuple[int, int] = (0, 0),
                 target_size: Optional[Tuple[int, int]] = None, unet_batch_one=False, prompt_embeds=None,
                 starting_image=None, strength=0.5, seed=None, rng="numpy", refiner_start=0.8, aesthetic_score=6.0,
                 negative_aesthetic_score=2.5, **kwargs):
        """``starting_image`` ((B, 3, H, W) in [-1, 1], the vae_encoder input) + ``strength`` select the Swift
        pipeline's image-to-image mode (StableDiffusionPipeline.swift:250-262, 361-378): the encoded image is noised
        to timestep ``timeSteps[startStep]`` and only the remaining steps run."""
        self.check_inputs(prompt, height, width, callback_steps)
        height = height or self.height
        width = width or self.width
        if (height, width) != (self.height, self.width):
            raise ValueError(f"this pipeline instance was built for {self.height}x{self.width} images")
        if eta < 0:
            raise ValueError(f"eta must be >= 0, got {eta}")
        if controlnet_cond and not self.controlnet:
            raise ValueError("Conditions for controlnet are given but the pipeline has no controlnet modules")
        prompts = [prompt] if isinstance(prompt, str) else list(prompt)
        prompts = [p for p in prompts for _ in range(num_images_per_prompt)]
        if len(prompts) != self.images_per_call:
            raise ValueError(f"this pipeline instance generates {self.images_per_call} image(s) per call, "
                             f"got {len(prompts)} prompt(s)")
        do_cfg = guidance_scale > 1.0  # pipeline.py:443
        xl_pooled = None
        if prompt_embeds is not None:
            text_embeddings = prompt_embeds
        elif self.xl and self.text_encoder_2 is not None:
            text_embeddings, xl_pooled = self._encode_prompt_xl(prompts, do_cfg, negative_prompt,
                                                                negative_prompt_2=kwargs.get("negative_prompt_2"))
        else:
            text_embeddings = self._encode_prompt(prompts, do_cfg, negative_prompt)
        time_ids = text_embeds = None
        if self.xl:
            original_size = original_size or (height, width)
            target_size = target_size or (height, width)
            ids = list(original_size) + list(crops_coords_top_left) + list(target_size)
            time_ids = torch.tensor([ids] * (2 * self.images_per_call), dtype=torch.float32, device=self.device)
            text_embeds = kwargs.get("pooled_prompt_embeds")
            if text_embeds is None and xl_pooled is not None:
                text_embeds = torch.as_tensor(xl_pooled, dtype=torch.float32, device=self.device)
            if text_embeds is None:
                text_embeds = torch.zeros(2 * self.images_per_call, 1280, device=self.device)
        lat = self.prepare_latents(len(prompts), self.unet.in_channels, height, width, latents, seed=seed, rng=rng)
        sched = self._make_scheduler(num_inference_steps, eta)
        start_step = 0
        if starting_image is None and sched.init_noise_sigma != 1.0:
            lat = lat * np.float32(sched.init_noise_sigma)  # pipeline.py:344 (sigma-space samplers)
        if starting_image is not None:
            if self.vae_encoder is None:
                raise ValueError("a starting image was provided but the pipeline has no vae_encoder")
            start_step = sched.start_step(strength)
            if start_step >= num_inference_steps:
                raise ValueError(f"strength {strength} leaves no denoising steps")
            # same draw order as the Swift pipeline: the noise samples first (above), then the encoder's noise
            enc_noise = np.random.randn(*lat.shape).astype(np.float32)
            x0 = self.vae_encoder.encode(np.asarray(starting_image, dtype=self.vae_encoder.expected_inputs["x"]["dtype"]),
                                         enc_noise, self.vae_decoder.engine.scaling).numpy()
            lat = sched.add_noise(x0.astype(np.float32), lat, strength)
        if controlnet_cond:  # pipeline.py:488-494
            controlnet_cond = self.prepare_control_cond(controlnet_cond, do_cfg, len(prompts), 1)
        refiner = None
        if self.unet_refiner is not None:
            # refiner conditioning (StableDiffusionXLPipeline.swift:314-345): the second encoder's embeddings only, its
            # pooled output, geometry = (original size, crop, aesthetic score) with the negative score on the uncond row
            r_emb = kwargs.get("refiner_prompt_embeds")
            r_pool = kwargs.get("refiner_pooled_prompt_embeds")
            if r_emb is None:
                if self.text_encoder_2 is None:
                    raise ValueError("the refiner needs text_encoder_2 or refiner_prompt_embeds / refiner_pooled_prompt_embeds")
                r_emb, r_pool = self._encode_prompt_xl(prompts, do_cfg, negative_prompt, only_second=True,
                                                       negative_prompt_2=kwargs.get("negative_prompt_2"))
            osz, crop = list(original_size or (height, width)), list(crops_coords_top_left)
            rows = [osz + crop + [negative_aesthetic_score]] * self.images_per_call + \
                   [osz + crop + [aesthetic_score]] * self.images_per_call
            refiner = {"encoder_hidden_states": r_emb, "text_embeds": torch.as_tensor(np.asarray(r_pool), dtype=torch.float32),
                       "time_ids": torch.tensor(rows, dtype=torch.float32)}
        final = self.denoise(text_embeddings, lat, num_inference_steps, guidance_scale, callback, callback_steps,
                             time_ids, text_embeds, controlnet_cond=controlnet_cond or None, start_step=start_step,
                             refiner=refiner, refiner_start=refiner_start, eta=eta, seed=seed)
        image = self.decode_latents(final).cpu().numpy()  # single device->host copy of the result
        has_nsfw = None  # the safety checker is out of scope (SURVEY section 2, row 19)
        if output_type == "pil":
            image = self.numpy_to_pil(image)
        if not return_dict:
            return (image, has_nsfw)
        return StableDiffusionPipelineOutput(images=image, nsfw_content_detected=has_nsfw)

    def generate(self, prompt, num_inference_steps=50, guidance_scale=7.5, **kwargs):
        """Alias named in BASELINE.json's north_star."""
        return self(prompt, num_inference_steps=num_inference_steps, guidance_scale=guidance_scale, **kwargs)
