"""Reverse-diffusion sampling — drop-in for ``tld.diffusion`` (reference tld/diffusion.py).

``DiffusionGenerator`` keeps the reference dataclass fields and the ``generate`` / ``pred_image`` /
``initialize_image`` / ``apply_classifier_free_guidance`` methods (tld/diffusion.py:22-125).  ``generate`` hands the
whole loop to ``tld_sampler_generate`` (include/tld_b200.h): the cond+uncond pair is packed in one 2B batch, the
conditioning K/V are hoisted out of the loop, and every diffusion step is one CUDA-graph replay.  ``edit_latents`` /
``edit`` (image-to-image, masked inpainting; ``outpaint_inputs`` for outpainting) run the same loop from partway down the
schedule through ``tld_sampler_edit`` (DESIGN.md §6d).

``DiffusionTransformer`` (tld/diffusion.py:143-186) is the text->image wrapper.  Its CLIP text tower and the
checkpoint download are pre-processing that needs third-party weights and network access; they are injected by
the caller (``text_encoder=`` / ``vae=``) instead of being pulled from the hub here.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import asdict, dataclass
from typing import Any, Callable, Optional

import numpy as np
import torch
from torch import Tensor

from . import _lib
from .configs import LTDConfig
from .denoiser import Denoiser
from .data import encode_image


def default_device() -> torch.device:
    return torch.device("cuda:0" if torch.cuda.is_available() else "cpu")


def noise_schedule(n_iter: int, exponent: float = 1, noise_levels=None) -> "list[float]":
    """Host-side schedule, computed exactly as tld/diffusion.py:50-52 (fp32 arange/pow -> python floats)."""
    if noise_levels is None:
        noise_levels = (1 - torch.pow(torch.arange(0, 1, 1 / n_iter), exponent)).tolist()
    noise_levels = list(noise_levels)
    noise_levels[0] = 0.99
    return noise_levels


def edit_schedule(n_iter: int, strength: float, exponent: float = 1, noise_levels=None) -> "tuple[list[float], int]":
    """Levels of an image-to-image / inpainting run: ``(noise_schedule(...)[i0:], i0)`` with
    ``i0 = min(round(n * (1 - strength)), n - 2)``, n the schedule's length (``n_iter`` unless ``noise_levels`` is given).
    ``strength = 1`` starts from pure noise (i0 = 0, first level 0.99); smaller strengths start partway down the schedule at
    the unmodified level ``sig[i0]``.  At least two levels (one update and the final prediction) always remain."""
    if not 0 < strength <= 1:
        raise ValueError(f"strength must be in (0, 1], got {strength}")
    sig = noise_schedule(n_iter, exponent, noise_levels)
    if len(sig) < 2:
        raise ValueError("need at least two noise levels")
    i0 = min(round(len(sig) * (1 - strength)), len(sig) - 2)
    return sig[i0:], i0


def outpaint_inputs(latent: Tensor, dx: int, dy: int) -> "tuple[Tensor, Tensor]":
    """Inputs for outpainting with the base model: the view moves ``dx`` latent pixels right and ``dy`` down (negative:
    left / up).  Returns ``(init_latents, mask)``: the latent shifted accordingly, zero in the uncovered band, and a
    ``[B,1,h,w]`` float32 mask that is 1 on that band (regenerate) and 0 where the old content is kept.  Pass both to
    ``DiffusionGenerator.edit_latents`` (strength 1); repeated calls extend a scene step by step."""
    if latent.dim() != 4:
        raise ValueError("outpaint_inputs: expected a latent [B,C,h,w]")
    B, _, h, w = latent.shape
    if not (abs(dx) < w and abs(dy) < h):
        raise ValueError(f"outpaint_inputs: shift ({dx}, {dy}) must be smaller than the latent ({w}, {h})")
    init = torch.zeros_like(latent)
    mask = torch.ones(B, 1, h, w, dtype=torch.float32, device=latent.device)
    # out[y, x] = latent[y + dy, x + dx] where that source pixel exists
    ys, xs = slice(max(0, -dy), h - max(0, dy)), slice(max(0, -dx), w - max(0, dx))
    yt, xt = slice(max(0, dy), h - max(0, -dy)), slice(max(0, dx), w - max(0, -dx))
    init[:, :, ys, xs] = latent[:, :, yt, xt]
    mask[:, :, ys, xs] = 0
    return init, mask


def _need_cuda_tensor(t: Tensor, what: str) -> None:
    if not isinstance(t, Tensor) or not t.is_cuda:
        raise _lib.TldError(f"{what}: CUDA tensor required (no CPU fallback)")
    if not t.is_floating_point():
        raise TypeError(f"{what}: floating-point tensor required, got {t.dtype}")


@dataclass
class DiffusionGenerator:
    model: Denoiser
    vae: Any  # anything with .decode(z) -> (image, ...) ; reference: diffusers.AutoencoderKL
    device: torch.device
    model_dtype: torch.dtype = torch.float32

    @torch.no_grad()
    def generate(
        self,
        labels: Tensor,
        n_iter: int = 30,
        num_imgs: int = 16,
        class_guidance: float = 3,
        seed: int = 10,
        scale_factor: int = 8,
        img_size: int = 32,
        sharp_f: float = 0.1,
        bright_f: float = 0.1,
        exponent: float = 1,
        seeds: Optional[Tensor] = None,
        noise_levels=None,
        use_ddpm_plus: bool = True,
    ):
        """Returns (decoded image on CPU, final latent on device) like tld/diffusion.py:29-92."""
        latent = self.generate_latents(labels, n_iter, num_imgs, class_guidance, seed, img_size, sharp_f, bright_f,
                                       exponent, seeds, noise_levels, use_ddpm_plus)
        img = self.vae.decode((latent * scale_factor).to(self.model_dtype))[0].cpu()
        return img, latent

    @torch.no_grad()
    def generate_grid_uint8(self, labels: Tensor, nrow: int, padding: int = 4, scale_factor: int = 8, **generate_kwargs):
        """Same sampling + decode as ``generate`` but the post-processing of tld/diffusion.py:185 / tld/train.py:36
        (``make_grid((out + 1) / 2, nrow, padding).clip(0, 1)`` -> ``ToPILImage``) runs on the device
        (``tld_image_grid_u8``) and only the finished uint8 HWC grid crosses PCIe: 1 byte per sample instead of 4
        (SURVEY.md §8(f) rank 3).  Returns (numpy uint8 [GH, GW, 3], final latent on device)."""
        latent = self.generate_latents(labels, **generate_kwargs)
        img = self.vae.decode((latent * scale_factor).to(self.model_dtype))[0]
        return image_grid_uint8(img, nrow, padding), latent

    @torch.no_grad()
    def generate_latents(self, labels: Tensor, n_iter: int = 30, num_imgs: int = 16, class_guidance: float = 3,
                         seed: int = 10, img_size: int = 32, sharp_f: float = 0.1, bright_f: float = 0.1,
                         exponent: float = 1, seeds: Optional[Tensor] = None, noise_levels=None,
                         use_ddpm_plus: bool = True) -> Tensor:
        """The sampling loop without the VAE decode (tld/diffusion.py:50-89) on the CUDA-graph sampler."""
        if torch.device(self.device).type != "cuda":
            raise _lib.TldError("DiffusionGenerator needs a CUDA device (no CPU fallback)")
        model = self.model
        if not isinstance(model, Denoiser):
            raise TypeError("DiffusionGenerator.model must be a transformer_latent_diffusion_b200.Denoiser")
        if img_size != model.image_size:
            raise ValueError(f"img_size={img_size} does not match the model's image_size={model.image_size}")
        sig = noise_schedule(n_iter, exponent, noise_levels)
        if len(sig) < 2:
            raise ValueError("need at least two noise levels")
        x_t = self.initialize_image(seeds, num_imgs, img_size, seed)
        if labels.shape[0] != num_imgs or x_t.shape[0] != num_imgs:
            raise ValueError("labels / seeds must have num_imgs rows")
        model.eval()
        dev = torch.device(self.device)
        h = model._ensure_handle(dev)
        lab = labels.to(device=dev, dtype=torch.float32).contiguous()
        x0 = x_t.to(device=dev, dtype=torch.float32).contiguous()
        out = torch.empty_like(x0)
        levels = (C.c_double * len(sig))(*sig)  # python floats, exactly as the reference loop sees them
        with torch.cuda.device(dev):
            _lib.check(_lib.load().tld_sampler_generate(
                h, _lib.ptr(lab), _lib.ptr(x0), _lib.ptr(out), num_imgs, levels, len(sig), float(class_guidance),
                float(sharp_f), float(bright_f), int(bool(use_ddpm_plus)), _lib.current_stream_ptr(dev)),
                "tld_sampler_generate")
        return out.to(self.model_dtype)

    @torch.no_grad()
    def edit_latents(self, labels: Tensor, init_latents: Tensor, strength: float = 1.0, mask: Optional[Tensor] = None,
                     n_iter: int = 30, class_guidance: float = 3, seed: int = 10, seeds: Optional[Tensor] = None,
                     exponent: float = 1, noise_levels=None, use_ddpm_plus: bool = True) -> Tensor:
        """Image-to-image and masked inpainting on the CUDA-graph sampler (``tld_sampler_edit``).

        ``init_latents`` [B,C,h,w] (CUDA) is the known latent in denoiser space (VAE latent / scale_factor).  The run
        covers ``edit_schedule(n_iter, strength, ...)``: strength 1 starts from the noise, a smaller strength from the known
        latent noised to the level it starts at.  ``mask`` (CUDA, [B,1,h,w] or [1,1,h,w], values clamped to [0, 1]):
        1 = regenerate, 0 = keep; the kept region follows the known latent re-noised with the same noise at every step and
        is returned unchanged.  The noise is drawn as in ``generate`` (``seed`` / ``seeds``).  Without a mask (or with an
        all-ones mask) and strength 1 the result is bit-identical to ``generate_latents(..., sharp_f=0, bright_f=0)``."""
        if torch.device(self.device).type != "cuda":
            raise _lib.TldError("DiffusionGenerator needs a CUDA device (no CPU fallback)")
        model = self.model
        if not isinstance(model, Denoiser):
            raise TypeError("DiffusionGenerator.model must be a transformer_latent_diffusion_b200.Denoiser")
        Cc, img = model.n_channels, model.image_size
        if init_latents.dim() != 4 or tuple(init_latents.shape[1:]) != (Cc, img, img):
            raise ValueError(f"edit_latents: init_latents must be [B,{Cc},{img},{img}], got {tuple(init_latents.shape)}")
        num_imgs = init_latents.shape[0]
        if labels.dim() != 2 or labels.shape[0] != num_imgs:
            raise ValueError("edit_latents: labels must have one row per init latent")
        if mask is not None and (mask.dim() != 4 or mask.shape[0] not in (1, num_imgs) or tuple(mask.shape[1:]) != (1, img, img)):
            raise ValueError(f"edit_latents: mask must be [B,1,{img},{img}] or [1,1,{img},{img}], got {tuple(mask.shape)}")
        _need_cuda_tensor(init_latents, "edit_latents: init_latents")
        if mask is not None:
            _need_cuda_tensor(mask, "edit_latents: mask")
        sig, i0 = edit_schedule(n_iter, strength, exponent, noise_levels)
        eps = self.initialize_image(seeds, num_imgs, img, seed)
        if tuple(eps.shape) != tuple(init_latents.shape):
            raise ValueError("edit_latents: seeds must have the init latents' shape")
        model.eval()
        dev = torch.device(self.device)
        h = model._ensure_handle(dev)
        lab = labels.to(device=dev, dtype=torch.float32).contiguous()
        noise = eps.to(device=dev, dtype=torch.float32).contiguous()
        x0k = init_latents.to(device=dev, dtype=torch.float32).contiguous()
        m = None if mask is None else mask.to(device=dev, dtype=torch.float32).expand(num_imgs, 1, img, img).contiguous()
        out = torch.empty_like(x0k)
        levels = (C.c_double * len(sig))(*sig)
        with torch.cuda.device(dev):
            _lib.check(_lib.load().tld_sampler_edit(
                h, _lib.ptr(lab), _lib.ptr(noise), _lib.ptr(x0k), None if m is None else _lib.ptr(m), _lib.ptr(out),
                num_imgs, levels, len(sig), int(i0 == 0), float(class_guidance), int(bool(use_ddpm_plus)),
                _lib.current_stream_ptr(dev)), "tld_sampler_edit")
        return out.to(self.model_dtype)

    def _edit_images(self, images01: Tensor, encoder, labels: Tensor, strength: float, mask: Optional[Tensor],
                     scale_factor: float, seed: int, seeds: Optional[Tensor], **kw) -> Tensor:
        # one device generator seeded with `seed` draws the posterior sample first, then the noise (unless seeds= is given)
        generator = torch.Generator(device=self.device)
        generator.manual_seed(seed)
        x0k = encode_image(images01, encoder, generator=generator, to_cpu=False).float() / scale_factor
        if seeds is None:
            seeds = torch.randn(x0k.shape, generator=generator, dtype=self.model_dtype, device=self.device)
        return self.edit_latents(labels, x0k, strength, mask, seeds=seeds, **kw)

    @torch.no_grad()
    def edit(self, images01: Tensor, encoder, labels: Tensor, strength: float = 1.0, mask: Optional[Tensor] = None,
             n_iter: int = 30, class_guidance: float = 3, seed: int = 10, seeds: Optional[Tensor] = None,
             exponent: float = 1, noise_levels=None, use_ddpm_plus: bool = True, scale_factor: int = 8):
        """Image-to-image / inpainting from pixels: ``images01`` [B,3,H,W] in [0, 1] is encoded with ``encoder`` (anything
        with ``.encode(x) -> (posterior,)``, e.g. ``vae.AutoencoderKLEncoder``) through ``data.encode_image``, the posterior
        sample divided by ``scale_factor`` is the known latent of ``edit_latents``.  A device generator seeded with ``seed``
        draws the posterior sample and then the noise.  ``mask`` is in latent resolution.  Returns (decoded image on CPU,
        final latent on device) like ``generate``."""
        latent = self._edit_images(images01, encoder, labels, strength, mask, scale_factor, seed, seeds, n_iter=n_iter,
                                   class_guidance=class_guidance, exponent=exponent, noise_levels=noise_levels,
                                   use_ddpm_plus=use_ddpm_plus)
        img = self.vae.decode((latent * scale_factor).to(self.model_dtype))[0].cpu()
        return img, latent

    def last_stats(self) -> "tuple[float, int]":
        """(device ms of the last sampling loop, kernel launches it issued)"""
        ms, n = C.c_float(), C.c_int64()
        _lib.check(_lib.load().tld_sampler_last_stats(self.model._ensure_handle(torch.device(self.device)),
                                                      C.byref(ms), C.byref(n)), "tld_sampler_last_stats")
        return ms.value, n.value

    @torch.no_grad()
    def pred_image(self, noisy_image: Tensor, labels: Tensor, noise_level: float, class_guidance: float) -> Tensor:
        """One CFG model call (tld/diffusion.py:94-103); `labels` is already cat[labels, zeros]."""
        num_imgs = noisy_image.size(0)
        noises = torch.full((2 * num_imgs, 1), noise_level)
        x0_pred = self.model(
            torch.cat([noisy_image, noisy_image]),
            noises.to(self.device, self.model_dtype),
            labels.to(self.device, self.model_dtype),
        )
        return self.apply_classifier_free_guidance(x0_pred, num_imgs, class_guidance)

    def initialize_image(self, seeds: Optional[Tensor], num_imgs: int, img_size: int, seed: int) -> Tensor:
        """Initial noise (tld/diffusion.py:105-120): device generator seeded with `seed`, or the given tensor."""
        if seeds is None:
            generator = torch.Generator(device=self.device)
            generator.manual_seed(seed)
            return torch.randn(num_imgs, self.model.n_channels, img_size, img_size, dtype=self.model_dtype,
                               device=self.device, generator=generator)
        return seeds.to(self.device, self.model_dtype)

    def apply_classifier_free_guidance(self, x0_pred: Tensor, num_imgs: int, class_guidance: float) -> Tensor:
        """tld/diffusion.py:122-125 — cond half first, uncond half second."""
        x0_pred_label, x0_pred_no_label = x0_pred[:num_imgs], x0_pred[num_imgs:]
        return class_guidance * x0_pred_label + (1 - class_guidance) * x0_pred_no_label


def make_image_grid(images: Tensor, nrow: int, padding: int = 4) -> Tensor:
    """(B,3,H,W) in [-1,1] -> one (3, H', W') grid in [0,1]; same layout as torchvision.utils.make_grid
    with pad value 0 (tld/diffusion.py:185), including its special case: a single image comes back unpadded."""
    imgs = ((images + 1) / 2).float()
    B, Cc, H, W = imgs.shape
    if B == 1:  # torchvision.utils.make_grid returns a single image as it is, without the padding frame
        return imgs[0].clip(0, 1)
    ncol = min(nrow, B)
    nrows = int(np.ceil(B / ncol))
    grid = imgs.new_zeros(Cc, nrows * (H + padding) + padding, ncol * (W + padding) + padding)
    for i in range(B):
        r, c = divmod(i, ncol)
        y, x = padding + r * (H + padding), padding + c * (W + padding)
        grid[:, y:y + H, x:x + W] = imgs[i]
    return grid.clip(0, 1)


def image_grid_uint8(images: Tensor, nrow: int, padding: int = 4) -> np.ndarray:
    """(B,3,H,W) in [-1,1] on the GPU -> uint8 [GH, GW, 3] numpy grid: bit-identical to
    ``(make_image_grid(images, nrow, padding).permute(1, 2, 0) * 255).byte()`` but computed by one CUDA kernel before the
    device-to-host copy."""
    if not images.is_cuda:
        raise _lib.TldError("image_grid_uint8: CUDA tensor required (no CPU fallback)")
    if images.dtype not in (torch.float32, torch.bfloat16):
        images = images.float()
    images = images.contiguous()
    B, Cc, H, W = images.shape
    if Cc != 3:
        raise ValueError("image_grid_uint8: expected RGB images [B,3,H,W]")
    ncol = min(nrow, B)
    nrows = -(-B // ncol)
    if B == 1:  # make_grid leaves a single image unpadded (the app's default num_imgs=1 must give an 8h x 8w image)
        padding = 0
    out = torch.empty(nrows * (H + padding) + padding, ncol * (W + padding) + padding, 3, dtype=torch.uint8,
                      device=images.device)
    _lib.check(_lib.load().tld_image_grid_u8(_lib.ptr(images), int(images.dtype == torch.bfloat16), _lib.ptr(out), B, H, W,
                                             ncol, padding, _lib.current_stream_ptr(images.device)), "tld_image_grid_u8")
    return out.cpu().numpy()


class DiffusionTransformer:
    """text -> image wrapper (tld/diffusion.py:143-186)."""

    def __init__(self, cfg: LTDConfig, vae: Any = None, text_encoder: Optional[Callable[[list], Tensor]] = None,
                 state_dict: Optional[dict] = None, device: Optional[torch.device] = None, encoder: Any = None):
        """``encoder`` (used by ``edit_image_from_text``): anything with ``.encode(x) -> (posterior,)``; by default the
        package's ``AutoencoderKLEncoder`` in ``cfg.vae_cfg.vae_dtype``, built on first use."""
        device = device or default_device()
        denoiser = Denoiser(**asdict(cfg.denoiser_cfg)).to(cfg.denoiser_load.dtype)
        if state_dict is None and cfg.denoiser_load.local_filename is not None:
            import os

            if os.path.exists(cfg.denoiser_load.local_filename):  # no network here: use the file if present
                state_dict = torch.load(cfg.denoiser_load.local_filename, map_location=torch.device("cpu"))
        if state_dict is not None:
            denoiser.load_state_dict(state_dict)
        denoiser = denoiser.to(device)
        if vae is None:
            from .vae import AutoencoderKLDecoder

            vae = AutoencoderKLDecoder().to(device=device, dtype=cfg.vae_cfg.vae_dtype)
        self.text_encoder = text_encoder
        self.encoder = encoder
        self._vae_dtype = cfg.vae_cfg.vae_dtype
        self.diffuser = DiffusionGenerator(denoiser, vae, device, cfg.denoiser_load.dtype)

    def generate_image_from_text(self, prompt: str, class_guidance=6, seed=11, num_imgs=1, img_size=32, n_iter=15):
        if self.text_encoder is None:
            raise _lib.TldError("no text encoder: pass text_encoder= (a callable prompt list -> [B,768] embeddings); "
                                "the CLIP ViT-L/14 tower is out of scope for this package")
        nrow = int(np.sqrt(num_imgs))
        labels = self.text_encoder([prompt] * num_imgs)
        arr, _ = self.diffuser.generate_grid_uint8(labels, nrow=nrow, padding=4, scale_factor=8, num_imgs=num_imgs,
                                                   img_size=self.diffuser.model.image_size, class_guidance=class_guidance,
                                                   seed=seed, n_iter=n_iter, exponent=1, sharp_f=0, bright_f=0)
        from PIL import Image

        return Image.fromarray(arr)

    def edit_image_from_text(self, prompt: str, image, mask=None, strength: float = 0.6, class_guidance=6, seed=11,
                             n_iter=15):
        """Image-to-image (``mask=None``) or inpainting / outpainting of a PIL ``image`` (RGB, side = 8 x the model's
        latent size) guided by ``prompt``.  ``mask``: a PIL image of the same size, non-zero = repaint; it is reduced to
        latent resolution by an 8x8 max-pool, so any repainted pixel repaints its whole latent pixel.  Returns a PIL image."""
        if self.text_encoder is None:
            raise _lib.TldError("no text encoder: pass text_encoder= (a callable prompt list -> [B,768] embeddings); "
                                "the CLIP ViT-L/14 tower is out of scope for this package")
        gen = self.diffuser
        side = 8 * gen.model.image_size
        if image.size != (side, side):
            raise ValueError(f"edit_image_from_text: image must be {side}x{side}, got {image.size[0]}x{image.size[1]}")
        img01 = torch.from_numpy(np.asarray(image.convert("RGB"), dtype=np.float32) / 255.0).permute(2, 0, 1)[None]
        m = None
        if mask is not None:
            if mask.size != image.size:
                raise ValueError("edit_image_from_text: mask and image must have the same size")
            pix = torch.from_numpy((np.asarray(mask.convert("L")) > 0).astype(np.float32))[None, None]
            m = torch.nn.functional.max_pool2d(pix, 8).to(gen.device)
        if self.encoder is None:
            from .vae import AutoencoderKLEncoder

            self.encoder = AutoencoderKLEncoder().to(device=gen.device, dtype=self._vae_dtype)
        labels = self.text_encoder([prompt])
        with torch.no_grad():
            latent = gen._edit_images(img01, self.encoder, labels, strength, m, 8, seed, None, n_iter=n_iter,
                                      class_guidance=class_guidance)
            out = gen.vae.decode((latent * 8).to(gen.model_dtype))[0]
        from PIL import Image

        return Image.fromarray(image_grid_uint8(out, nrow=1, padding=4))
