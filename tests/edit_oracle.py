"""fp32 statement of image-to-image / masked inpainting on the reference sampler loop.  TEST INFRASTRUCTURE ONLY.

The reference has no edit loop; this states the package's semantics (``include/tld_b200.h:tld_sampler_edit``, DESIGN.md
§6d) with the oracle's unmodified building blocks (``noise_schedule``, ``multistep_ratios``, ``cfg_combine``,
``denoiser_forward``), next to its ``generate_latents``, so that the edit tests compare the CUDA sampler with it.
"""
from __future__ import annotations

import torch

from oracle.tld_oracle import OracleCfg, cfg_combine, denoiser_forward, multistep_ratios, noise_schedule


def edit_latents(sd, cfg: OracleCfg, labels: torch.Tensor, init_latents: torch.Tensor, noise: torch.Tensor,
                 strength: float = 1.0, mask=None, n_iter: int = 30, class_guidance: float = 3, exponent: float = 1,
                 noise_levels=None, use_ddpm_plus: bool = True) -> torch.Tensor:
    """Image-to-image / masked inpainting on the reference loop (not in the reference; the package's
    ``tld_sampler_edit``).  ``init_latents`` = known latent x0k (VAE latent / scale factor), ``noise`` = eps,
    ``mask`` [B or 1,1,h,w]: 1 = regenerate, 0 = keep.

    1. schedule: sig = noise_schedule(...) ([0] = 0.99), i0 = min(round(n (1 - strength)), n - 2), run over sig[i0:]
    2. start: x = eps if i0 == 0, else sig[i0] eps + (1 - sig[i0]) x0k (the training corruption, tld/train.py:130)
    3. loop: tld/diffusion.py:66-85 over the truncated list, ratios from that list, first step first order
    4. with a mask, after each update to level nxt: x = m x + (1 - m) (nxt eps + (1 - nxt) x0k), the same eps every step
    5. out = m x0 + (1 - m) x0k (x0 without a mask); no sharp / bright shifts
    """
    if not 0 < strength <= 1:
        raise ValueError(f"strength must be in (0, 1], got {strength}")
    sig = noise_schedule(n_iter, exponent, noise_levels)
    i0 = min(round(len(sig) * (1 - strength)), len(sig) - 2)
    sig = sig[i0:]
    rs = multistep_ratios(sig) if use_ddpm_plus else None
    x0k, eps = init_latents, noise
    num = x0k.shape[0]
    m = None if mask is None else mask.clamp(0, 1).expand(num, 1, *x0k.shape[2:])
    x_t = eps.clone() if i0 == 0 else sig[0] * eps + (1 - sig[0]) * x0k
    lab2 = torch.cat([labels, torch.zeros_like(labels)])

    def pred(xt, s):
        t = torch.full((2 * num, 1), s, dtype=xt.dtype, device=xt.device)
        return cfg_combine(denoiser_forward(sd, cfg, torch.cat([xt, xt]), t, lab2), num, class_guidance)

    prev = None
    nxt = sig[0]
    for i in range(len(sig) - 1):
        cur, nxt = sig[i], sig[i + 1]
        x0 = pred(x_t, cur)
        if prev is None or not use_ddpm_plus:
            d = x0
        else:
            d = (1 + 1 / (2 * rs[i - 1])) * x0 - (1 / (2 * rs[i - 1])) * prev
        x_t = ((cur - nxt) * d + nxt * x_t) / cur
        if m is not None:
            x_t = m * x_t + (1 - m) * (nxt * eps + (1 - nxt) * x0k)
        prev = x0
    x0 = pred(x_t, nxt)
    return x0 if m is None else m * x0 + (1 - m) * x0k
