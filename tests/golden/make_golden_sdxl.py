"""Golden fixture for BASELINE configs[3]: SDXL-base UNet (UNet2DConditionModelXL, 2.57 B parameters) at 768x768
(96x96 latents), produced by the UNMODIFIED reference modules on the CPU in fp32 (about 10 GB of RAM, a few
minutes):

    B200SD_REFERENCE=<reference checkout> python tests/golden/make_golden_sdxl.py

Weights are regenerated from the seed on the test side (see make_golden.py); stored: the inputs that are not
seed-derived, the reference output and a weight fingerprint.
"""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from b200sd import config  # noqa: E402
from oracle import ref_unet  # noqa: E402
from make_golden import fingerprint, unet_inputs  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def main():
    cfg = config.SDXL_BASE_UNET
    t0 = time.time()
    sd = config.random_state_dict(config.unet_param_shapes(cfg), seed=31, dtype=torch.float16)
    x, c = unet_inputs(cfg, 32, size=96)
    g = torch.Generator().manual_seed(33)
    te = torch.randn(2, 1280, generator=g)
    tid = torch.tensor([[768.0, 768.0, 0.0, 0.0, 768.0, 768.0]] * 2)
    m = ref_unet.build_unet(cfg, sd, xl=True, impl="SPLIT_EINSUM")
    print(f"built in {time.time() - t0:.0f} s")
    t0 = time.time()
    with torch.no_grad():
        y = m(x.half().float(), torch.tensor([981.0, 981.0]), c.half().float(), tid, te.half().float())[0].numpy()
    print(f"forward {time.time() - t0:.0f} s, absmax {np.abs(y).max():.4f}, std {y.std():.4f}")
    np.savez_compressed(os.path.join(OUT, "unet_sdxl_768.npz"), weight_seed=31, input_seed=32, embed_seed=33,
                        fingerprint=fingerprint(sd), time_ids=tid.numpy(), noise_pred=y.astype(np.float32))


if __name__ == "__main__":
    main()
