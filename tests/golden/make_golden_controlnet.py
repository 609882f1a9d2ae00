"""Golden fixture for BASELINE configs[4]: the SD-2.1 ControlNet (361 M parameters) at 64x64 latents / 512x512
condition image, produced by the UNMODIFIED reference module (python_coreml_stable_diffusion/controlnet.py) on the
CPU in fp32:

    B200SD_REFERENCE=<reference checkout> python tests/golden/make_golden_controlnet.py

The 13 residuals are stored at fp16 precision with a fixed spatial stride to keep the fixture under 1 MB; weights
are regenerated from the seed on the test side (see make_golden.py).
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from b200sd import config  # noqa: E402
from oracle import ref_unet  # noqa: E402
from make_golden import fingerprint, unet_inputs  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
STRIDE = 8  # residuals are sub-sampled [:, :, ::STRIDE, ::STRIDE]


def main():
    cfg = config.SD21_CONTROLNET
    sd = config.random_state_dict(config.controlnet_param_shapes(cfg), seed=51, dtype=torch.float16)
    x, c = unet_inputs(config.SD21_BASE_UNET, 52)
    cond = torch.rand(2, 3, 512, 512, generator=torch.Generator().manual_seed(53))
    cn = ref_unet.build_controlnet(cfg, sd)
    with torch.no_grad():
        down, mid = cn(x.half().float(), torch.tensor([501.0, 501.0]), c.half().float(), cond.half().float())
    res = list(down) + [mid]
    print([tuple(r.shape) for r in res], [round(float(r.abs().max()), 3) for r in res])
    np.savez_compressed(os.path.join(OUT, "controlnet_sd21.npz"), weight_seed=51, input_seed=52, cond_seed=53,
                        stride=STRIDE, fingerprint=fingerprint(sd),
                        **{f"residual_{i}": r[:, :, ::STRIDE, ::STRIDE].numpy().astype(np.float16) for i, r in enumerate(res)})


if __name__ == "__main__":
    main()
