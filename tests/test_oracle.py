"""CPU tests that pin the oracle (oracle/restated.py) and the engine's parameter schemas against the golden
fixtures produced by the unmodified reference modules (tests/golden/make_golden*.py)."""
import gzip
import json
import os

import numpy as np
import pytest
import torch

from b200sd import config
from oracle import restated as R

GOLD = os.path.join(os.path.dirname(__file__), "golden")
sys_path_inserted = True


def _load(name):
    return np.load(os.path.join(GOLD, name))


def _reference_schema(name):
    """{parameter name: shape} of the reference module built from config.<name>."""
    with gzip.open(os.path.join(GOLD, "param_schemas.json.gz"), "rt") as f:
        return {k: tuple(v) for k, v in json.load(f)[name].items()}


def _fingerprint(sd):
    keys = sorted(sd.keys())
    picks = [keys[0], keys[len(keys) // 2], keys[-1]]
    return np.array([float(sd[k].double().sum()) for k in picks] + [float(len(keys))])


def _inputs(cfg, seed, batch=2, seq=77):
    g = torch.Generator().manual_seed(seed)
    s = cfg["sample_size"]
    x = torch.randn(batch, cfg["in_channels"], s, s, generator=g)
    c = torch.randn(batch, cfg["cross_attention_dim"], 1, seq, generator=g)
    return x, c


@pytest.mark.parametrize("name,cfg", [("tiny", config.TINY_UNET), ("sd21", config.SD21_BASE_UNET)])
def test_restated_unet_matches_reference_golden(name, cfg):
    gold = _load(f"unet_{name}.npz")
    sd = config.random_state_dict(config.unet_param_shapes(cfg), seed=int(gold["weight_seed"]))
    assert np.allclose(_fingerprint(sd), gold["fingerprint"], rtol=1e-6), "weight generator drifted"
    x, c = _inputs(cfg, int(gold["input_seed"]))
    t = torch.tensor([float(gold["timestep"])] * 2)
    with torch.no_grad():
        y = R.unet_forward(sd, cfg, x, t, c).numpy()
    for key in gold.files:
        if key.startswith("noise_pred_"):
            assert np.abs(y - gold[key]).max() < 2e-5, key
            assert R.compute_psnr(torch.from_numpy(y), torch.from_numpy(gold[key])) > 100


def test_restated_xl_and_controlnet_match_reference_golden():
    gold = _load("unet_tiny_xl.npz")
    cfg = config.TINY_XL_UNET
    sd = config.random_state_dict(config.unet_param_shapes(cfg), seed=int(gold["weight_seed"]))
    assert np.allclose(_fingerprint(sd), gold["fingerprint"], rtol=1e-6)
    x, c = _inputs(cfg, int(gold["input_seed"]))
    with torch.no_grad():
        y = R.unet_forward(sd, cfg, x, torch.tensor([981.0, 981.0]), c, time_ids=torch.from_numpy(gold["time_ids"]),
                           text_embeds=torch.from_numpy(gold["text_embeds"])).numpy()
    assert np.abs(y - gold["noise_pred"]).max() < 2e-5
    gold = _load("controlnet_tiny.npz")
    ccfg = config.TINY_CONTROLNET
    csd = config.random_state_dict(config.controlnet_param_shapes(ccfg), seed=int(gold["weight_seed"]))
    assert np.allclose(_fingerprint(csd), gold["fingerprint"], rtol=1e-6)
    x, c = _inputs(config.TINY_UNET, int(gold["input_seed"]))
    cond = torch.rand(2, 3, 128, 128, generator=torch.Generator().manual_seed(int(gold["cond_seed"])))
    with torch.no_grad():
        outs = R.controlnet_forward(csd, ccfg, x, torch.tensor([501.0, 501.0]), c, cond)
    assert len(outs) == 7
    for i, o in enumerate(outs):
        assert np.abs(o.numpy() - gold[f"residual_{i}"]).max() < 2e-5, i


def test_controlnet_schema_matches_reference_modules():
    for name in ("TINY_CONTROLNET", "SD21_CONTROLNET"):
        ref_shapes = _reference_schema(name)
        mine = {k: tuple(v) for k, v in config.controlnet_param_shapes(getattr(config, name)).items()}
        assert ref_shapes == mine, (name, set(ref_shapes.items()) ^ set(mine.items()))


def _block_inputs(seed):
    """The operands make_golden.block_inputs drew for blocks.npz."""
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(2, 128, 1, 200, generator=g)
    k = torch.randn(2, 128, 1, 77, generator=g)
    v = torch.randn(2, 128, 1, 77, generator=g)
    w = torch.randn(128, generator=g)
    b = torch.randn(128, generator=g)
    mask = torch.zeros(2, 77, 1, 1)
    mask[:, 50:] = -1e4
    return q, k, v, mask, w, b


def test_restated_blocks_match_reference_golden():
    g = _load("blocks.npz")
    q, k, v, mask, w, b = _block_inputs(int(g["input_seed"]))
    fp = np.array([float(t.double().sum()) for t in (q, k, v, w, b)])
    assert np.allclose(fp, g["input_fingerprint"], rtol=1e-6), "input generator drifted"
    ref = R.attention(q, k, v, 2, 64).numpy()
    for nm in ("original", "split_einsum", "split_einsum_v2"):
        assert np.abs(ref - g[f"attn_{nm}"]).max() < 2e-6, nm
    masked = R.attention(q, k, v, 2, 64, mask=mask).numpy()
    assert np.abs(masked - g["attn_split_einsum_masked"]).max() < 2e-6
    # LayerNormANE is (x_hat + b) * w; the oracle/engine convention is x_hat * w + b' with b' = b * w
    ln = R.layer_norm_channels(q, w, b * w).numpy()
    assert np.abs(ln - g["ln_out"]).max() < 2e-5
    temb = R.timestep_embedding(torch.tensor([981.0, 1.0, 500.0]), 320).numpy()
    assert np.abs(temb - g["temb"]).max() < 1e-6


def test_param_schema_matches_reference_modules():
    for name in ("TINY_UNET", "SD21_BASE_UNET", "SDXL_BASE_UNET"):
        ref_shapes = _reference_schema(name)
        mine = {k: tuple(v) for k, v in config.unet_param_shapes(getattr(config, name)).items()}
        assert ref_shapes == mine, (name, set(ref_shapes.items()) ^ set(mine.items()))


def test_restated_matches_live_reference_tiny_all_impls():
    """Tiny UNet with a different timestep per batch row against the reference's output under each of its three
    attention implementations (unet_tiny_timesteps.npz)."""
    gold = _load("unet_tiny_timesteps.npz")
    cfg = config.TINY_UNET
    sd = config.random_state_dict(config.unet_param_shapes(cfg), seed=int(gold["weight_seed"]))
    assert np.allclose(_fingerprint(sd), gold["fingerprint"], rtol=1e-6), "weight generator drifted"
    x, c = _inputs(cfg, int(gold["input_seed"]))
    t = torch.from_numpy(gold["timesteps"])
    with torch.no_grad():
        y = R.unet_forward(sd, cfg, x, t, c).numpy()
    for impl in ("ORIGINAL", "SPLIT_EINSUM", "SPLIT_EINSUM_V2"):
        assert np.abs(y - gold[f"noise_pred_{impl}"]).max() < 2e-5, impl


def test_compute_psnr_definition():
    a = torch.tensor([1.0, -2.0, 3.0])
    b = torch.tensor([1.0, -2.0, 3.5])
    rmse = (0.25 / 3) ** 0.5
    assert abs(R.compute_psnr(a, b) - 20 * np.log10((3.5 + 1e-5) / (rmse + 1e-10))) < 1e-9
    assert R.compute_psnr(a, a) > 200


def test_vae_decoder_restatement_shapes_and_postprocess():
    cfg = config.TINY_VAE
    sd = config.random_state_dict(config.vae_decoder_param_shapes(cfg), seed=3)
    z = torch.randn(1, 4, 8, 8)
    with torch.no_grad():
        img = R.vae_decode(sd, cfg, z)
    assert img.shape == (1, 3, 32, 32) and torch.isfinite(img).all()
    pp = R.postprocess_image(img)
    assert pp.shape == (1, 32, 32, 3) and pp.min() >= 0 and pp.max() <= 1
    # linear-in-last-conv identity: scaling conv_out weights+bias scales the image
    sd2 = dict(sd)
    sd2["decoder.conv_out.weight"] = sd["decoder.conv_out.weight"] * 2
    sd2["decoder.conv_out.bias"] = sd["decoder.conv_out.bias"] * 2
    with torch.no_grad():
        assert torch.allclose(R.vae_decode(sd2, cfg, z), 2 * img, atol=1e-5)


@pytest.mark.parametrize("cfg_name", ["TINY_CLIP_TEXT", "CLIP_L_TEXT"])
def test_clip_text_restatement_matches_transformers(cfg_name):
    """The text-encoder restatement against the library class the reference converts (transformers.CLIPTextModel)."""
    from b200sd import config
    from oracle import clip_text

    if not clip_text.available():
        pytest.skip("transformers not importable")
    cfg = dict(getattr(config, cfg_name))
    if cfg_name == "CLIP_L_TEXT":
        cfg["num_hidden_layers"] = 2  # quick_gelu path; two layers keep the CPU test fast
    sd = config.random_clip_text_state_dict(cfg, seed=5)
    ids = torch.randint(0, cfg["vocab_size"], (2, 77), generator=torch.Generator().manual_seed(6))
    ids[:, -1] = cfg["vocab_size"] - 1
    ref = clip_text.library_forward(cfg, sd, ids)
    out = clip_text.clip_text_forward(cfg, sd, ids)
    assert out.shape == ref.shape == (2, 77, cfg["hidden_size"])
    assert float((out - ref).abs().max()) < 2e-5


@pytest.mark.parametrize("cfg_name", ["TINY_CLIP_TEXT", "TINY_CLIP_TEXT_PROJ"])
def test_clip_text_hidden_states_and_pooled_match_transformers(cfg_name):
    """hidden_states[-2] / pooler_output / text_embeds: the tensors torch2coreml.py:416-433 exports for SDXL."""
    from b200sd import config
    from oracle import clip_text

    if not clip_text.available():
        pytest.skip("transformers not importable")
    cfg = getattr(config, cfg_name)
    sd = config.random_clip_text_state_dict(cfg, seed=9)
    ids = torch.randint(0, cfg["vocab_size"] - 2, (3, 77), generator=torch.Generator().manual_seed(10))
    ids[0, 5:] = cfg["vocab_size"] - 1
    ids[1, 76] = cfg["vocab_size"] - 1
    ids[2, 30] = cfg["vocab_size"] - 1
    ref = clip_text.library_forward_all(cfg, sd, ids)
    out = clip_text.clip_text_forward(cfg, sd, ids, return_all=True)
    assert len(out["hidden_states"]) == len(ref["hidden_states"]) == cfg["num_hidden_layers"] + 1
    assert float((out["hidden_states"][-2] - ref["hidden_states"][-2]).abs().max()) < 2e-5
    assert float((out["last_hidden_state"] - ref["last_hidden_state"]).abs().max()) < 2e-5
    key = "text_embeds" if cfg.get("projection_dim") else "pooler_output"
    assert out[key].shape == ref[key].shape and float((out[key] - ref[key]).abs().max()) < 2e-5


def test_restated_controlnet_sd21_matches_reference_golden():
    """BASELINE configs[4] network at full size (361 M parameters, 512x512 condition image): the restatement
    against the residuals of the unmodified reference module (tests/golden/make_golden_controlnet.py)."""
    gold = _load("controlnet_sd21.npz")
    cfg = config.SD21_CONTROLNET
    sd = config.random_state_dict(config.controlnet_param_shapes(cfg), seed=int(gold["weight_seed"]), dtype=torch.float16)
    g = torch.Generator().manual_seed(int(gold["input_seed"]))
    x = torch.randn(2, 4, 64, 64, generator=g)
    c = torch.randn(2, 1024, 1, 77, generator=g)
    cond = torch.rand(2, 3, 512, 512, generator=torch.Generator().manual_seed(int(gold["cond_seed"])))
    st = int(gold["stride"])
    with torch.no_grad():
        outs = R.controlnet_forward(sd, cfg, x.half().float(), torch.tensor([501.0, 501.0]), c.half().float(),
                                    cond.half().float())
    assert len(outs) == 13
    for i, o in enumerate(outs):
        ref = torch.from_numpy(gold[f"residual_{i}"].astype(np.float32))
        err = float((o[:, :, ::st, ::st] - ref).abs().max())
        assert err < 2e-3 * max(1.0, float(ref.abs().max())), (i, err)  # the fixture is stored in fp16
