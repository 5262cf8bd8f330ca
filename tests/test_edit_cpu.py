"""Image-to-image / inpainting without a GPU: the edit schedule, the oracle's edit loop against its generate loop, the
outpainting helper and the argument checks of DiffusionGenerator.edit_latents."""
import math

import pytest
import torch

from oracle import tld_oracle as O

import edit_oracle as E
from transformer_latent_diffusion_b200 import _lib
from transformer_latent_diffusion_b200.diffusion import DiffusionGenerator, edit_schedule, outpaint_inputs


@pytest.mark.parametrize("n_iter,exponent", [(2, 1), (3, 1), (15, 1), (30, 1), (35, 2.0), (50, 1)])
def test_edit_schedule_is_a_tail_of_the_generate_schedule(n_iter, exponent):
    full = O.noise_schedule(n_iter, exponent)
    strengths = [k / 200 for k in range(1, 201)] + [1e-9, 0.5 / n_iter, 1 - 1e-9]
    for s in strengths:
        levels, i0 = edit_schedule(n_iter, s, exponent)
        assert i0 == min(round(n_iter * (1 - s)), n_iter - 2)
        assert levels == full[i0:], (s, i0)
        assert len(levels) >= 2
    levels, i0 = edit_schedule(n_iter, 1.0, exponent)
    assert i0 == 0 and levels == full and levels[0] == 0.99


def test_edit_schedule_custom_levels():
    custom = [0.9, 0.7, 0.5, 0.3, 0.1]
    levels, i0 = edit_schedule(30, 0.6, noise_levels=custom)   # n is the length of the given list
    assert i0 == 2 and levels == [0.5, 0.3, 0.1]


@pytest.mark.parametrize("bad", [0.0, -0.25, 1.0001, 2.0, math.nan])
def test_edit_schedule_rejects_bad_strength(bad):
    with pytest.raises(ValueError):
        edit_schedule(30, bad)
    with pytest.raises(ValueError):
        E.edit_latents({}, O.OracleCfg(), torch.zeros(1, 768), torch.zeros(1, 4, 16, 16), torch.zeros(1, 4, 16, 16),
                       strength=bad)


@pytest.fixture(scope="module")
def tiny():
    cfg = O.OracleCfg(image_size=8, embed_dim=64, n_layers=1)
    sd = O.synth_state_dict(cfg, 11)
    g = torch.Generator().manual_seed(12)
    labels = torch.randn(2, 768, generator=g)
    eps = torch.randn(2, 4, 8, 8, generator=g)
    x0k = torch.randn(2, 4, 8, 8, generator=g) * 0.5
    return cfg, sd, labels, eps, x0k


@pytest.mark.parametrize("ddpm_plus", [True, False])
def test_oracle_edit_at_strength_1_is_generate(tiny, ddpm_plus):
    cfg, sd, labels, eps, x0k = tiny
    kw = dict(n_iter=6, class_guidance=4.0, use_ddpm_plus=ddpm_plus)
    with torch.no_grad():
        gen = O.generate_latents(sd, cfg, labels, eps, sharp_f=0, bright_f=0, **kw)
        plain = E.edit_latents(sd, cfg, labels, x0k, eps, strength=1.0, **kw)
        ones = E.edit_latents(sd, cfg, labels, x0k, eps, strength=1.0, mask=torch.ones(1, 1, 8, 8), **kw)
        zeros = E.edit_latents(sd, cfg, labels, x0k, eps, strength=0.6, mask=torch.zeros(2, 1, 8, 8), **kw)
    assert torch.equal(plain, gen) and torch.equal(ones, gen)
    assert torch.equal(zeros, x0k)


def test_oracle_edit_keeps_the_masked_out_region(tiny):
    cfg, sd, labels, eps, x0k = tiny
    mask = torch.zeros(2, 1, 8, 8)
    mask[..., 4:] = 1.0
    with torch.no_grad():
        out = E.edit_latents(sd, cfg, labels, x0k, eps, strength=0.6, mask=mask, n_iter=6)
        free = E.edit_latents(sd, cfg, labels, x0k, eps, strength=0.6, n_iter=6)
    assert torch.equal(out[..., :4], x0k[..., :4])
    assert not torch.equal(out[..., 4:], free[..., 4:])   # the kept half steers the regenerated half


@pytest.mark.parametrize("dx,dy", [(3, 0), (-2, 0), (0, 5), (-1, -4), (6, 2), (0, 0)])
def test_outpaint_inputs_geometry(dx, dy):
    lat = torch.arange(2 * 4 * 8 * 10, dtype=torch.float32).reshape(2, 4, 8, 10) + 1   # no zeros: the band is visible
    init, mask = outpaint_inputs(lat, dx, dy)
    assert init.shape == lat.shape and mask.shape == (2, 1, 8, 10) and mask.dtype == torch.float32
    for y in range(8):
        for x in range(10):
            sy, sx = y + dy, x + dx
            if 0 <= sy < 8 and 0 <= sx < 10:
                assert torch.equal(init[:, :, y, x], lat[:, :, sy, sx]) and (mask[:, :, y, x] == 0).all()
            else:
                assert (init[:, :, y, x] == 0).all() and (mask[:, :, y, x] == 1).all()


def test_outpaint_inputs_rejects_bad_shifts():
    lat = torch.zeros(1, 4, 8, 8)
    for dx, dy in [(8, 0), (0, -8), (9, 9)]:
        with pytest.raises(ValueError):
            outpaint_inputs(lat, dx, dy)
    with pytest.raises(ValueError):
        outpaint_inputs(torch.zeros(4, 8, 8), 1, 0)


def test_edit_latents_refuses_cpu_tensors_and_wrong_shapes():
    from transformer_latent_diffusion_b200.denoiser import Denoiser

    m = Denoiser(16, 256, 2, 128, 0, 1)
    gen = DiffusionGenerator(m, None, torch.device("cuda:0"), torch.float32)   # nothing here touches a device
    lab = torch.zeros(2, 768)
    with pytest.raises(_lib.TldError):
        gen.edit_latents(lab, torch.zeros(2, 4, 16, 16))                        # CPU init latents
    for bad in [torch.zeros(2, 4, 8, 8), torch.zeros(2, 3, 16, 16), torch.zeros(4, 16, 16)]:
        with pytest.raises(ValueError):
            gen.edit_latents(lab, bad)
    with pytest.raises(ValueError):
        gen.edit_latents(torch.zeros(3, 768), torch.zeros(2, 4, 16, 16))        # labels row count
    for bad in [torch.zeros(2, 4, 16, 16), torch.zeros(3, 1, 16, 16), torch.zeros(2, 1, 8, 8), torch.zeros(16, 16)]:
        with pytest.raises(ValueError):
            gen.edit_latents(lab, torch.zeros(2, 4, 16, 16), mask=bad)
    with pytest.raises(_lib.TldError):
        DiffusionGenerator(m, None, torch.device("cpu")).edit_latents(lab, torch.zeros(2, 4, 16, 16))
