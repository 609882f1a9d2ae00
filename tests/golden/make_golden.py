"""Generates the golden fixtures under tests/golden/ by running the UNMODIFIED reference modules
(python_coreml_stable_diffusion.{unet,attention,layer_norm,controlnet}) imported through oracle/ref_unet.py
from a checkout of apple/ml-stable-diffusion:

    B200SD_REFERENCE=<reference checkout> python tests/golden/make_golden.py [fixture ...]

With no argument every fixture below is rewritten; otherwise only the named ones (see FIXTURES).
Weights are not stored: they are regenerated from a seed by b200sd.config.random_state_dict (CPU
torch generator, deterministic for a given torch build); a fingerprint of them is stored so a
generator mismatch is detected instead of silently failing parity.
"""
import gzip
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from b200sd import config  # noqa: E402
from oracle import ref_unet  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def fingerprint(sd):
    keys = sorted(sd.keys())
    picks = [keys[0], keys[len(keys) // 2], keys[-1]]
    return np.array([float(sd[k].double().sum()) for k in picks] + [float(len(keys))])


def unet_inputs(cfg, seed, batch=2, seq=77, size=None):
    g = torch.Generator().manual_seed(seed)
    s = size or cfg["sample_size"]
    x = torch.randn(batch, cfg["in_channels"], s, s, generator=g)
    c = torch.randn(batch, cfg["cross_attention_dim"], 1, seq, generator=g)
    return x, c


def block_inputs(seed=5):
    """Attention / LayerNormANE operands of blocks.npz (regenerated from the seed by the test as well)."""
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(2, 128, 1, 200, generator=g)
    k = torch.randn(2, 128, 1, 77, generator=g)
    v = torch.randn(2, 128, 1, 77, generator=g)
    ln_w = torch.randn(128, generator=g)
    ln_b = torch.randn(128, generator=g)
    mask = torch.zeros(2, 77, 1, 1)
    mask[:, 50:] = -1e4
    return q, k, v, mask, ln_w, ln_b


def unets():
    """Full UNet, three attention implementations, tiny + SD-2.1-base."""
    for name, cfg, wseed, iseed, t in [("tiny", config.TINY_UNET, 1, 2, 981.0),
                                       ("sd21", config.SD21_BASE_UNET, 1, 2, 981.0)]:
        sd = config.random_state_dict(config.unet_param_shapes(cfg), seed=wseed)
        x, c = unet_inputs(cfg, iseed)
        ts = torch.tensor([t, t])
        outs = {}
        for impl in ("ORIGINAL", "SPLIT_EINSUM", "SPLIT_EINSUM_V2"):
            if name == "sd21" and impl != "ORIGINAL":
                continue
            m = ref_unet.build_unet(cfg, sd, impl=impl)
            with torch.no_grad():
                outs[impl] = m(x, ts, c)[0].numpy()
        np.savez_compressed(os.path.join(OUT, f"unet_{name}.npz"), weight_seed=wseed, input_seed=iseed,
                            timestep=t, fingerprint=fingerprint(sd),
                            **{f"noise_pred_{k}": v.astype(np.float32) for k, v in outs.items()})
        print(name, {k: float(np.abs(v).max()) for k, v in outs.items()})


def unet_tiny_timesteps():
    """Tiny UNet at two different timesteps per batch row, all three attention implementations."""
    cfg = config.TINY_UNET
    sd = config.random_state_dict(config.unet_param_shapes(cfg), seed=7)
    x, c = unet_inputs(cfg, 8)
    t = torch.tensor([501.0, 21.0])
    outs = {}
    for impl in ("ORIGINAL", "SPLIT_EINSUM", "SPLIT_EINSUM_V2"):
        m = ref_unet.build_unet(cfg, sd, impl=impl)
        with torch.no_grad():
            outs[impl] = m(x, t, c)[0].numpy().astype(np.float32)
    np.savez_compressed(os.path.join(OUT, "unet_tiny_timesteps.npz"), weight_seed=7, input_seed=8,
                        timesteps=t.numpy(), fingerprint=fingerprint(sd),
                        **{f"noise_pred_{k}": v for k, v in outs.items()})
    print("tiny timesteps", {k: float(np.abs(v).max()) for k, v in outs.items()})


def xl_and_controlnet():
    """SDXL-style UNet (UNet2DConditionModelXL) and ControlNetModel, tiny configs."""
    cfg = config.TINY_XL_UNET
    sd = config.random_state_dict(config.unet_param_shapes(cfg), seed=3)
    x, c = unet_inputs(cfg, 9)
    gg = torch.Generator().manual_seed(10)
    tid = torch.tensor([[64.0, 64.0, 0.0, 0.0, 64.0, 64.0]] * 2)
    te = torch.randn(2, 64, generator=gg)
    m = ref_unet.build_unet(cfg, sd, xl=True, impl="SPLIT_EINSUM")
    with torch.no_grad():
        y = m(x, torch.tensor([981.0, 981.0]), c, tid, te)[0].numpy()
    np.savez_compressed(os.path.join(OUT, "unet_tiny_xl.npz"), weight_seed=3, input_seed=9, fingerprint=fingerprint(sd),
                        text_embeds=te.numpy(), time_ids=tid.numpy(), noise_pred=y.astype(np.float32))
    ccfg = config.TINY_CONTROLNET
    csd = config.random_state_dict(config.controlnet_param_shapes(ccfg), seed=4)
    x, c = unet_inputs(config.TINY_UNET, 6)
    cond = torch.rand(2, 3, 128, 128, generator=torch.Generator().manual_seed(7))
    cn = ref_unet.build_controlnet(ccfg, csd)
    with torch.no_grad():
        down, mid = cn(x.clone(), torch.tensor([501.0, 501.0]), c, cond)
    np.savez_compressed(os.path.join(OUT, "controlnet_tiny.npz"), weight_seed=4, input_seed=6, cond_seed=7,
                        fingerprint=fingerprint(csd),
                        **{f"residual_{i}": r.numpy().astype(np.float32) for i, r in enumerate(list(down) + [mid])})
    print("xl + controlnet done")


def blocks():
    """Attention variants + LayerNormANE + timestep embedding on their own.  The operands are not stored (see
    block_inputs); a fingerprint of them is."""
    ref = ref_unet.load()
    q, k, v, mask, ln_w, ln_b = block_inputs()
    att = {}
    for nm, fn in (("original", ref.attention.original), ("split_einsum", ref.attention.split_einsum),
                   ("split_einsum_v2", ref.attention.split_einsum_v2)):
        att[nm] = fn(q.clone(), k.clone(), v.clone(), None, 2, 64).numpy()
    att["split_einsum_masked"] = ref.attention.split_einsum(q.clone(), k.clone(), v.clone(), mask, 2, 64).numpy()
    ln = ref.layer_norm.LayerNormANE(128)
    with torch.no_grad():
        ln.weight.copy_(ln_w)
        ln.bias.copy_(ln_b)
        ln_out = ln(q.clone()).numpy()
    temb = ref.unet.get_timestep_embedding(torch.tensor([981.0, 1.0, 500.0]), 320, flip_sin_to_cos=True,
                                           downscale_freq_shift=0).numpy()
    inputs_fp = np.array([float(t.double().sum()) for t in (q, k, v, ln_w, ln_b)])
    np.savez_compressed(os.path.join(OUT, "blocks.npz"), input_seed=5, input_fingerprint=inputs_fp, ln_out=ln_out,
                        temb=temb, **{f"attn_{k_}": v_ for k_, v_ in att.items()})
    print("blocks done")


def schemas():
    """Parameter names and shapes of the reference UNet / ControlNet modules for every config the engine builds."""
    out = {}
    for name, xl in (("TINY_UNET", False), ("SD21_BASE_UNET", False), ("SDXL_BASE_UNET", True)):
        with torch.device("meta"):
            m = ref_unet.build_unet(getattr(config, name), None, xl=xl)
        out[name] = {k: list(v.shape) for k, v in m.state_dict().items()}
    for name in ("TINY_CONTROLNET", "SD21_CONTROLNET"):
        with torch.device("meta"):
            m = ref_unet.build_controlnet(getattr(config, name))
        out[name] = {k: list(v.shape) for k, v in m.state_dict().items()}
    # mtime=0: the same schemas give the same bytes
    with gzip.GzipFile(os.path.join(OUT, "param_schemas.json.gz"), "wb", mtime=0) as f:
        f.write(json.dumps(out, sort_keys=True).encode())
    print("schemas", {k: len(v) for k, v in out.items()})


FIXTURES = {"unets": unets, "unet_tiny_timesteps": unet_tiny_timesteps, "xl_and_controlnet": xl_and_controlnet,
            "blocks": blocks, "schemas": schemas}


def main(names):
    torch.manual_seed(0)
    ref_unet.load()
    for name in names or FIXTURES:
        FIXTURES[name]()


if __name__ == "__main__":
    main(sys.argv[1:])
