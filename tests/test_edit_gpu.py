"""Image-to-image and masked inpainting on the CUDA-graph sampler (tld_sampler_edit) against the sampler itself, the oracle's
edit loop (tests/edit_oracle.py) and the library's VAE encoder / decoder.

Bars: bit-identity where the arithmetic is the same (strength 1 without a mask or with an all-ones mask is the generate loop;
the kept region is the known latent), rel-Fro < 3e-2 on the regenerated region against the fp32 oracle (the multi-step
sampler bar of tests/test_forward_gpu.py), 2e-2 for the headline 100M configuration.
"""
import numpy as np
import pytest
import torch

from conftest import rel_fro
from oracle import tld_oracle as O

import edit_oracle as E

pytestmark = pytest.mark.gpu


def _model(cfg: O.OracleCfg, sd):
    from transformer_latent_diffusion_b200.denoiser import Denoiser

    m = Denoiser(cfg.image_size, cfg.noise_embed_dims, cfg.patch_size, cfg.embed_dim, cfg.dropout, cfg.n_layers,
                 cfg.text_emb_size, cfg.mlp_multiplier, cfg.n_channels)
    m.load_state_dict(sd, strict=True)
    return m.cuda().eval()


def _setup(img, D, L, B, seed):
    from transformer_latent_diffusion_b200.diffusion import DiffusionGenerator

    from oracle.ref_loader import IdentityVAE

    cfg = O.OracleCfg(image_size=img, embed_dim=D, n_layers=L)
    sd = O.synth_state_dict(cfg, seed)
    gen = DiffusionGenerator(_model(cfg, sd), IdentityVAE(), torch.device("cuda:0"), torch.float32)
    g = torch.Generator().manual_seed(seed + 1)
    labels = torch.randn(B, 768, generator=g)
    eps = torch.randn(B, 4, img, img, generator=g)
    x0k = 0.5 * torch.randn(B, 4, img, img, generator=g)
    return cfg, sd, gen, labels, eps, x0k


def _half_mask(B, img):
    m = torch.zeros(B, 1, img, img)
    m[..., img // 2:] = 1.0
    return m


@pytest.mark.parametrize("img,D,L,B", [(16, 128, 2, 3), (32, 256, 2, 2)])
@pytest.mark.parametrize("ddpm_plus", [True, False])
def test_strength_1_is_generate_bit_for_bit(img, D, L, B, ddpm_plus):
    cfg, sd, gen, labels, eps, x0k = _setup(img, D, L, B, 101)
    kw = dict(n_iter=8, class_guidance=4.0, use_ddpm_plus=ddpm_plus)
    ref = gen.generate_latents(labels, num_imgs=B, img_size=img, seeds=eps, sharp_f=0, bright_f=0, **kw)
    plain = gen.edit_latents(labels, x0k.cuda(), 1.0, seeds=eps, **kw)
    ones = gen.edit_latents(labels, x0k.cuda(), 1.0, mask=torch.ones(1, 1, img, img, device="cuda"), seeds=eps, **kw)
    assert torch.equal(plain, ref)
    assert torch.equal(ones, ref)


def test_zero_mask_returns_the_known_latent():
    cfg, sd, gen, labels, eps, x0k = _setup(16, 128, 2, 3, 111)
    for strength in (0.3, 1.0):
        out = gen.edit_latents(labels, x0k.cuda(), strength, mask=torch.zeros(3, 1, 16, 16, device="cuda"), n_iter=8,
                               seeds=eps)
        assert torch.equal(out.cpu(), x0k)


@pytest.mark.parametrize("img,D,L,B", [(16, 128, 2, 3), (32, 256, 2, 2)])   # the second: fused 256-token kernels
def test_edit_vs_oracle(img, D, L, B):
    cfg, sd, gen, labels, eps, x0k = _setup(img, D, L, B, 121)
    g = torch.Generator().manual_seed(122)
    binary = (torch.rand(B, 1, img, img, generator=g) < 0.5).float()
    soft = torch.rand(B, 1, img, img, generator=g) * 1.6 - 0.3          # values outside [0, 1]: clamped on both sides
    soft[..., : img // 4] = 0.0                                          # and a band kept exactly
    for strength in (0.3, 0.6, 1.0):
        for mask in (None, binary, soft):
            for ddpm_plus in (True, False):
                kw = dict(n_iter=10, class_guidance=4.0, use_ddpm_plus=ddpm_plus)
                out = gen.edit_latents(labels, x0k.cuda(), strength, None if mask is None else mask.cuda(), seeds=eps,
                                       **kw).cpu()
                with torch.no_grad():
                    ref = E.edit_latents(sd, cfg, labels, x0k, eps, strength, mask, **kw)
                what = (strength, None if mask is None else ("binary" if mask is binary else "soft"), ddpm_plus)
                regen = torch.ones_like(out, dtype=torch.bool) if mask is None else (mask.clamp(0, 1) > 0).expand_as(out)
                assert rel_fro(out[regen], ref[regen]) < 3e-2, (what, rel_fro(out[regen], ref[regen]))
                if mask is not None:
                    assert torch.equal(out[~regen], x0k[~regen]), what


def test_edit_refuses_a_cpu_mask():
    from transformer_latent_diffusion_b200 import _lib

    cfg, sd, gen, labels, eps, x0k = _setup(16, 128, 1, 2, 131)
    with pytest.raises(_lib.TldError):
        gen.edit_latents(labels, x0k.cuda(), 0.5, mask=torch.ones(2, 1, 16, 16), n_iter=4, seeds=eps)


def test_headline_config_half_mask_vs_oracle():
    """100M model, 32x32 latent (256 px), 35 steps, guidance 6, B 2, strength 0.6, right half regenerated."""
    cfg, sd, gen, labels, eps, x0k = _setup(32, 768, 12, 2, 141)
    mask = _half_mask(2, 32)
    kw = dict(n_iter=35, class_guidance=6.0)
    out = gen.edit_latents(labels, x0k.cuda(), 0.6, mask.cuda(), seeds=eps, **kw).cpu()
    torch.set_num_threads(max(1, min(32, (torch.get_num_threads() or 1))))
    with torch.no_grad():
        ref = E.edit_latents(sd, cfg, labels, x0k, eps, 0.6, mask, **kw)
    err = rel_fro(out[..., 16:], ref[..., 16:])
    assert err < 2e-2, f"strength 0.6 half-mask 100M edit rel_fro={err:.3e}"
    assert torch.equal(out[..., :16], x0k[..., :16])


def test_generate_and_edit_graphs_do_not_disturb_each_other():
    """The masked edit has its own captured graph; both graphs bake in the sampler buffers, so a reallocation for a larger
    batch must drop both (a stale masked graph would read freed buffers)."""
    cfg, sd, gen, labels, eps, x0k = _setup(16, 128, 2, 3, 151)
    mask = _half_mask(3, 16).cuda()
    g = torch.Generator().manual_seed(152)
    labels5, eps5 = torch.randn(5, 768, generator=g), torch.randn(5, 4, 16, 16, generator=g)
    kw = dict(n_iter=8, class_guidance=4.0)

    def generate(lab=labels, e=eps):
        return gen.generate_latents(lab, num_imgs=lab.shape[0], img_size=16, seeds=e, **kw).clone()

    def edit(m=mask, strength=0.6):
        return gen.edit_latents(labels, x0k.cuda(), strength, m, seeds=eps, **kw).clone()

    gen_a = generate()
    masked_a = edit()
    plain_a = edit(None)
    gen_b = generate()
    assert torch.equal(gen_a, gen_b)
    assert torch.equal(edit(), masked_a) and torch.equal(edit(None), plain_a)
    generate(labels5, eps5)                      # larger batch: the sampler buffers move
    assert torch.equal(edit(), masked_a)
    assert torch.equal(edit(None), plain_a)
    assert torch.equal(generate(), gen_a)
    assert not torch.equal(masked_a, plain_a)


def test_last_stats_count_one_start_kernel_more_than_generate():
    from transformer_latent_diffusion_b200.diffusion import edit_schedule

    cfg, sd, gen, labels, eps, x0k = _setup(16, 128, 2, 3, 161)
    mask = _half_mask(3, 16).cuda()
    for strength in (1.0, 0.6):
        levels, _ = edit_schedule(12, strength)
        gen.generate_latents(labels, num_imgs=3, img_size=16, seeds=eps, noise_levels=levels)
        ms_g, n_gen = gen.last_stats()
        for m in (None, mask):
            gen.edit_latents(labels, x0k.cuda(), strength, m, n_iter=12, seeds=eps)
            ms, n = gen.last_stats()
            assert ms > 0 and n == n_gen + 1, (strength, m is None, n, n_gen)


class _EncodeOnce(torch.nn.Module):
    """The library's VAE encoder, run once per input image batch.  Its GroupNorm statistics are summed with shared-memory
    atomics in no fixed order, so two encodes of the same batch may differ in the last bits; returning the posterior of the
    first run lets the test rebuild the exact known latent the edit used."""

    def __init__(self, enc):
        super().__init__()
        self.enc = enc
        self.last = None
        self.runs = 0

    def encode(self, x, return_dict=False):
        if self.last is None or not torch.equal(self.last[0], x):
            self.last = (x.clone(), self.enc.encode(x, return_dict=return_dict))
            self.runs += 1
        return self.last[1]


def test_edit_end_to_end_on_the_library_vae():
    """DiffusionGenerator.edit at 256 px (32x32 latent) with a right-half mask on the library's encoder and decoder: the kept
    half is the posterior sample / 8 bit for bit; edit_image_from_text returns a 256x256 PIL image."""
    from PIL import Image

    from transformer_latent_diffusion_b200.configs import DenoiserConfig, DenoiserLoad, LTDConfig
    from transformer_latent_diffusion_b200.data import encode_image
    from transformer_latent_diffusion_b200.diffusion import DiffusionGenerator, DiffusionTransformer
    from transformer_latent_diffusion_b200.vae import AutoencoderKLDecoder, AutoencoderKLEncoder

    torch.manual_seed(0)
    enc = _EncodeOnce(AutoencoderKLEncoder().cuda().to(torch.bfloat16).eval())
    dec = AutoencoderKLDecoder().cuda().to(torch.bfloat16).eval()
    cfg = O.OracleCfg(image_size=32, embed_dim=256, n_layers=2)
    gen = DiffusionGenerator(_model(cfg, O.synth_state_dict(cfg, 171)), dec, torch.device("cuda:0"), torch.float32)
    g = torch.Generator().manual_seed(172)
    images = torch.rand(2, 3, 256, 256, generator=g).cuda()
    labels = torch.randn(2, 768, generator=g)
    mask = _half_mask(1, 32).cuda()
    img, lat = gen.edit(images, enc, labels, strength=0.6, mask=mask, n_iter=10, seed=5)
    assert img.device.type == "cpu" and img.shape == (2, 3, 256, 256) and torch.isfinite(img).all()
    assert lat.is_cuda and lat.shape == (2, 4, 32, 32)
    x0k = encode_image(images, enc, generator=torch.Generator(device="cuda").manual_seed(5), to_cpu=False).float() / 8
    assert enc.runs == 1
    assert torch.equal(lat[..., :16], x0k[..., :16])
    assert not torch.equal(lat[..., 16:], x0k[..., 16:])

    def fake_clip(prompts):
        return torch.randn(len(prompts), 768, generator=g).cuda()

    ltd = LTDConfig(denoiser_cfg=DenoiserConfig(image_size=32, n_layers=1),
                    denoiser_load=DenoiserLoad(file_url=None, local_filename=None))
    dt = DiffusionTransformer(ltd, vae=dec, text_encoder=fake_clip, device=torch.device("cuda:0"), encoder=enc.enc)
    rgb = (np.random.default_rng(0).random((256, 256, 3)) * 255).astype(np.uint8)
    pmask = np.zeros((256, 256), dtype=np.uint8)
    pmask[:, 128:] = 255
    out = dt.edit_image_from_text("a cyberpunk marketplace", Image.fromarray(rgb), Image.fromarray(pmask), n_iter=6)
    assert isinstance(out, Image.Image) and out.size == (256, 256)
    out2 = dt.edit_image_from_text("a cyberpunk marketplace", Image.fromarray(rgb), n_iter=6)   # image-to-image
    assert out2.size == (256, 256)


def test_backward_pending_across_an_edit_is_refused():
    from transformer_latent_diffusion_b200 import _lib
    from transformer_latent_diffusion_b200.diffusion import DiffusionGenerator

    from oracle.ref_loader import IdentityVAE

    cfg = O.OracleCfg(image_size=16, embed_dim=128, n_layers=1)
    m = _model(cfg, O.synth_state_dict(cfg, 181))
    gen = DiffusionGenerator(m, IdentityVAE(), torch.device("cuda:0"), torch.float32)
    g = torch.Generator().manual_seed(182)
    x, t, lab = torch.randn(2, 4, 16, 16, generator=g).cuda(), torch.rand(2, 1, generator=g).cuda(), torch.randn(2, 768, generator=g).cuda()
    for mask in (None, _half_mask(2, 16).cuda()):
        a = m.train()(x, t, lab)
        gen.edit_latents(lab, x * 0.5, 0.6, mask, n_iter=4)
        with pytest.raises(_lib.TldError):
            a.square().mean().backward()
    a = m.train()(x, t, lab)
    a.square().mean().backward()
    assert all(p.grad is not None for p in m.parameters())
