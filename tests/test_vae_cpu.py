"""CPU suite for the first-stage decoder (SURVEY.md §8f N1): the oracle restatement against the
outputs of the reference's own `Decoder` / `Encoder` (recorded by oracle/make_golden_ref.py) and against the
reference-generated golden vectors; the host-side graph of editanything_b200.vae with the operators
emulated on CPU (tests/cpu_ops.py); the diffusers -> ldm key map."""
import os

import pytest
import torch

from editanything_b200.vae import DiagonalGaussian, VaeDecoderEngine, VaeEncoderEngine, VaeEngine
from editanything_b200.vae_spec import (SD_VAE, VAE_TINY, make_vae_state_dict, vae_decoder_param_shapes,
                                        vae_encoder_param_shapes)
from editanything_b200.weights import vae_diffusers_to_ldm, vae_ldm_to_diffusers_names
from oracle import vae_oracle as V
from oracle.make_golden_vae import make_image, make_latents
from tests import cpu_ops

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_param_count_matches_kl_f8_decoder():
    n = 0
    for shape, _ in vae_decoder_param_shapes(SD_VAE).values():
        k = 1
        for s in shape:
            k *= s
        n += k
    assert abs(n - 49.49e6) < 0.05e6, n      # SURVEY.md §8a R17: 49.5 M parameters


def test_oracle_matches_reference_decoder():
    cfg = VAE_TINY
    sd = make_vae_state_dict(cfg, 21)
    z = make_latents(cfg, 2, 12, 5) / cfg.scaling_factor
    ref = torch.load(os.path.join(GOLD, "ref_vae_modules.pt"))["decoded"]      # the reference's Decoder(z)
    with torch.no_grad():
        ours = V.decode(z, sd, cfg)
    assert ours.shape == ref.shape and (ours - ref).abs().max().item() < 2e-5


def test_oracle_reproduces_reference_golden():
    g = torch.load(os.path.join(GOLD, "vae_tiny.pt"))
    m = g["meta"]
    sd = make_vae_state_dict(VAE_TINY, m["weight_seed"])
    with torch.no_grad():
        img = V.decode_latents(make_latents(VAE_TINY, m["B"], m["side"], m["latent_seed"]), sd, VAE_TINY)
    assert (img - g["image"]).abs().max().item() < 2e-5


def test_host_graph_matches_golden_with_emulated_ops():
    g = torch.load(os.path.join(GOLD, "vae_tiny.pt"))
    m = g["meta"]
    sd = make_vae_state_dict(VAE_TINY, m["weight_seed"])
    eng = VaeDecoderEngine(VAE_TINY, {"first_stage_model." + k: v for k, v in sd.items()}, torch.device("cpu"),
                           backend=cpu_ops)
    lat = make_latents(VAE_TINY, m["B"], m["side"], m["latent_seed"])
    img = eng.decode_latents(lat)
    assert img.shape == g["image"].shape and img.dtype == torch.float32
    assert (img - g["image"]).abs().max().item() < 5e-4
    raw = eng.decode(lat / VAE_TINY.scaling_factor).sample          # the `vae.decode(z).sample` contract
    c = raw.shape[2] // 2
    assert (raw[:, :, c - 8:c + 8, c - 8:c + 8] - g["raw_center"]).abs().max().item() < 2e-3
    assert eng.config.scaling_factor == VAE_TINY.scaling_factor and len(eng.config.block_out_channels) == 2


def test_rejects_wrong_latent_channels():
    sd = make_vae_state_dict(VAE_TINY, 3)
    eng = VaeDecoderEngine(VAE_TINY, sd, torch.device("cpu"), backend=cpu_ops)
    with pytest.raises(ValueError):
        eng.decode_latents(torch.zeros(1, 3, 8, 8))


def test_diffusers_key_map_round_trip():
    sd = make_vae_state_dict(SD_VAE, 1, dtype=torch.float16)
    names = vae_ldm_to_diffusers_names(SD_VAE)
    assert set(names) == set(sd)
    dsd = {names[k]: (v.reshape(v.shape[0], v.shape[1]) if ".attentions." in names[k] and v.dim() == 4 else v)
           for k, v in sd.items()}
    assert "decoder.up_blocks.0.resnets.0.conv1.weight" in dsd and "decoder.mid_block.attentions.0.to_q.weight" in dsd
    back = vae_diffusers_to_ldm(dsd, SD_VAE)
    assert set(back) == set(sd)
    for k in sd:
        assert back[k].shape == sd[k].shape and torch.equal(back[k], sd[k]), k


# ---- encode side ------------------------------------------------------------------------------------
def test_param_count_matches_kl_f8_encoder():
    n = 0
    for shape, _ in vae_encoder_param_shapes(SD_VAE).values():
        k = 1
        for s in shape:
            k *= s
        n += k
    assert abs(n - 34.16e6) < 0.05e6, n      # SURVEY.md §8a R6: 34.2 M parameters


def test_encode_oracle_matches_reference_encoder():
    cfg = VAE_TINY
    sd = make_vae_state_dict(cfg, 31, part="encoder")
    x = make_image(2, 24, 6)              # odd spatial size after the stride-2: exercises the (0,1,0,1) padding
    ref = torch.load(os.path.join(GOLD, "ref_vae_modules.pt"))["moments"]      # the reference's Encoder(x)
    with torch.no_grad():
        ours = V.encode_moments(x, sd, cfg)
    assert ours.shape == ref.shape and (ours - ref).abs().max().item() < 2e-5


def test_encode_oracle_reproduces_reference_golden():
    g = torch.load(os.path.join(GOLD, "vae_enc_tiny.pt"))
    m = g["meta"]
    sd = make_vae_state_dict(VAE_TINY, m["weight_seed"], part="encoder")
    with torch.no_grad():
        mom = V.encode_moments(make_image(m["B"], m["side"], m["image_seed"]), sd, VAE_TINY)
    assert (mom - g["moments"]).abs().max().item() < 2e-5


def test_encoder_host_graph_matches_golden_with_emulated_ops():
    g = torch.load(os.path.join(GOLD, "vae_enc_tiny.pt"))
    m = g["meta"]
    sd = make_vae_state_dict(VAE_TINY, m["weight_seed"], part="encoder")
    eng = VaeEncoderEngine(VAE_TINY, sd, torch.device("cpu"), backend=cpu_ops)
    dist = eng.encode(make_image(m["B"], m["side"], m["image_seed"])).latent_dist
    ref = DiagonalGaussian(g["moments"])
    assert (dist.mean - ref.mean).abs().max().item() < 1e-3 and (dist.logvar - ref.logvar).abs().max().item() < 1e-3
    # latent_dist.sample(generator): mean + std * randn drawn from the caller's generator (reproducible)
    s1 = dist.sample(generator=torch.Generator().manual_seed(5))
    s2 = dist.sample(generator=torch.Generator().manual_seed(5))
    noise = torch.randn(dist.mean.shape, generator=torch.Generator().manual_seed(5))
    assert torch.equal(s1, s2) and torch.allclose(s1, dist.mean + dist.std * noise)
    assert torch.equal(dist.mode(), dist.mean)
    with pytest.raises(ValueError):
        eng.encode(torch.zeros(1, 4, 32, 32))
    with pytest.raises(ValueError):
        eng.encode(torch.zeros(1, 3, 33, 32))


def test_full_engine_round_trip_surface():
    """VaeEngine = encode + decode + decode_latents + config behind one object (what `pipe.vae` is)."""
    sd = dict(make_vae_state_dict(VAE_TINY, 1, part="encoder"))
    sd.update(make_vae_state_dict(VAE_TINY, 2))
    eng = VaeEngine(VAE_TINY, sd, torch.device("cpu"), backend=cpu_ops)
    z = eng.encode(make_image(1, 32, 3)).latent_dist.mode() * eng.config.scaling_factor
    assert z.shape == (1, 4, 16, 16)
    img = eng.decode_latents(z)
    assert img.shape == (1, 3, 32, 32) and float(img.min()) >= 0.0 and float(img.max()) <= 1.0


def test_encoder_diffusers_key_map_round_trip():
    sd = make_vae_state_dict(SD_VAE, 1, dtype=torch.float16, part="encoder")
    names = vae_ldm_to_diffusers_names(SD_VAE, part="encoder")
    assert set(names) == set(sd)
    dsd = {names[k]: (v.reshape(v.shape[0], v.shape[1]) if ".attentions." in names[k] and v.dim() == 4 else v)
           for k, v in sd.items()}
    assert "encoder.down_blocks.0.downsamplers.0.conv.weight" in dsd and "encoder.conv_norm_out.weight" in dsd
    back = vae_diffusers_to_ldm(dsd, SD_VAE, parts=("encoder",))
    assert set(back) == set(sd) and all(torch.equal(back[k], sd[k]) for k in sd)

