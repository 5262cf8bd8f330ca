#!/usr/bin/env python3
"""Per-step device time of the masked edit against plain generation at the 100M config (256 px, random weights).

Alternates generate_latents and a masked edit_latents (strength 1, right half regenerated: the same number of steps as
generate) in one process, ROUNDS times each, and prints one JSON object: ms per step of every round from the sampler's own
CUDA events (last_stats), median and spread (max - min) per arm, launch counts, and the device name and power limit read in
the same run.  The masked update reads the known latent, the noise and the mask on top of the plain update: about 2.4 MB per
step at batch 64.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import torch

from transformer_latent_diffusion_b200.denoiser import Denoiser
from transformer_latent_diffusion_b200.diffusion import DiffusionGenerator


class _Id:
    def decode(self, z):
        return (z,)


def _power_limit() -> str:
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--img", type=int, default=32)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--steps", type=int, default=35)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_edit.py needs a CUDA device")
    torch.manual_seed(0)
    m = Denoiser(a.img, 256, 2, 768, 0, 12).cuda().eval()
    gen = DiffusionGenerator(m, _Id(), torch.device("cuda:0"), torch.float32)
    labels = torch.randn(a.batch, 768, device="cuda")
    seeds = torch.randn(a.batch, 4, a.img, a.img, device="cuda")
    x0k = torch.randn(a.batch, 4, a.img, a.img, device="cuda")
    mask = torch.zeros(1, 1, a.img, a.img, device="cuda")
    mask[..., a.img // 2:] = 1.0
    arms = {
        "generate": lambda: gen.generate_latents(labels, n_iter=a.steps, num_imgs=a.batch, img_size=a.img, seeds=seeds,
                                                 class_guidance=6, sharp_f=0, bright_f=0),
        "masked_edit": lambda: gen.edit_latents(labels, x0k, 1.0, mask, n_iter=a.steps, class_guidance=6, seeds=seeds),
    }
    for f in arms.values():   # capture both step graphs and warm up
        f()
    torch.cuda.synchronize()
    per_step = {k: [] for k in arms}
    launches = {}
    for _ in range(a.rounds):
        for k, f in arms.items():
            f()
            ms, n = gen.last_stats()
            per_step[k].append(ms / a.steps)
            launches[k] = n
    res = {
        "device": torch.cuda.get_device_name(0),
        "power_limit": _power_limit(),
        "config": {"model": "100M (D 768, 12 layers)", "latent": a.img, "batch": a.batch, "steps": a.steps,
                   "mask": "right half", "strength": 1.0, "weights": "random"},
        "ms_per_step": {k: [round(v, 4) for v in vs] for k, vs in per_step.items()},
        "median_ms_per_step": {k: round(sorted(vs)[len(vs) // 2], 4) for k, vs in per_step.items()},
        "spread_ms_per_step": {k: round(max(vs) - min(vs), 4) for k, vs in per_step.items()},
        "launches": launches,
    }
    print(json.dumps(res))


if __name__ == "__main__":
    main()
