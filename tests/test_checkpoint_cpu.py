"""Real-checkpoint path on the CPU (no GPU work: instantiation, key routing, config round trip, channel surgery)."""
import os

import pytest
import torch

from conftest import GOLD
from gligen_b200 import checkpoint as CK
from gligen_b200.pipeline import GROUNDING_INPUT, model_config
from gligen_b200.spec import NAMED_CONFIGS, NAMED_VAE_CONFIGS, synthetic_state_dict, synthetic_vae_encoder_state_dict, synthetic_vae_state_dict


def _config(name="tiny", vae="tiny_vae64"):
    cfg, v = NAMED_CONFIGS[name], NAMED_VAE_CONFIGS[vae]
    dd = dict(double_z=True, z_channels=v.z_channels, resolution=v.image_size, in_channels=3, out_ch=v.out_ch, ch=v.ch, ch_mult=list(v.ch_mult),
              num_res_blocks=v.num_res_blocks, attn_resolutions=[], dropout=0.0)
    return {"model": model_config(cfg),
            "autoencoder": {"target": "ldm.models.autoencoder.AutoencoderKL", "params": dict(ddconfig=dd, embed_dim=v.embed_dim, scale_factor=v.scale_factor)},
            "diffusion": {"target": "ldm.models.diffusion.ldm.LatentDiffusion", "params": dict(linear_start=0.00085, linear_end=0.012, timesteps=1000)},
            "grounding_tokenizer_input": {"target": GROUNDING_INPUT[cfg.tokenizer]}}


def test_checkpoint_round_trip(tmp_path):
    """save (reference layout: config_dict._content + four state dicts) -> load_ckpt: classes located by their dotted names,
    the 966-key-style UNet state dict loads strictly, a full VAE state dict (with encoder keys) is accepted."""
    cfg, v = NAMED_CONFIGS["tiny"], NAMED_VAE_CONFIGS["tiny_vae64"]
    sd = synthetic_state_dict(cfg, 0)
    vsd = dict(synthetic_vae_state_dict(v, 0))
    vsd.update(synthetic_vae_encoder_state_dict(v, 1))          # a real checkpoint carries both halves (encoder.* / quant_conv.*)
    path = os.path.join(str(tmp_path), "gligen.pth")
    from ldm.models.diffusion.ldm import LatentDiffusion
    dsd = LatentDiffusion(linear_start=0.00085, linear_end=0.012, timesteps=1000).state_dict()      # schedule buffers, as in a real checkpoint
    from gligen_b200.clip_text import TINY_CLIP_TEXT, synthetic_clip_state_dict
    cfg_all = _config()
    cfg_all["text_encoder"] = {"target": "ldm.modules.encoders.modules.FrozenCLIPEmbedder", "params": {"text_config": "tiny_clip_text"}}
    tsd = synthetic_clip_state_dict(TINY_CLIP_TEXT, 0)
    tsd["transformer.text_model.embeddings.position_ids"] = torch.arange(77)[None]          # buffer older transformers releases save
    CK.save_ckpt(path, cfg_all, sd, autoencoder_sd=vsd, text_encoder_sd=tsd, diffusion_sd=dsd)
    model, vae, text, diffusion, config = CK.load_ckpt(path, device="cpu", with_text_encoder=False)
    assert type(model).__module__ == "ldm.modules.diffusionmodules.openaimodel" and text is None
    _, _, text, _, _ = CK.load_ckpt(path, device="cpu")
    k = "transformer.text_model.encoder.layers.1.self_attn.q_proj.weight"
    assert type(text).__module__ == "ldm.modules.encoders.modules" and torch.equal(text.state_dict()[k], tsd[k])
    got = model.state_dict()
    assert set(got) == set(sd) and all(torch.equal(got[k], sd[k]) for k in sd)
    assert model.grounding_tokenizer_input is not None and hasattr(model.grounding_tokenizer_input, "prepare")
    vgot = vae.state_dict()
    assert set(vgot) == set(vsd) and all(torch.equal(vgot[k], vsd[k]) for k in vsd)
    assert diffusion.num_timesteps == 1000 and config["model"]["target"].endswith("UNetModel")


def test_inpaint_channel_surgery_matches_reference():
    """add_additional_channels == the reference's convert_ckpt.add_additional_channels on a 320-channel first conv, and the widened
    state dict loads into the inpainting UNet (9 input channels, openaimodel.py:299-305)."""
    g = torch.Generator().manual_seed(0)
    w = torch.randn(320, 4, 3, 3, generator=g)
    mine = {"input_blocks.0.0.weight": w.clone(), "other": torch.ones(2)}
    CK.add_additional_channels(mine, 5)
    assert mine["input_blocks.0.0.weight"].shape == (320, 9, 3, 3) and torch.equal(mine["input_blocks.0.0.weight"][:, :4], w)
    assert mine["input_blocks.0.0.weight"][:, 4:].abs().sum() == 0 and torch.equal(mine["other"], torch.ones(2))
    # the reference's result on the same seeded weight (oracle/gen_golden_small.py)
    gold = torch.load(os.path.join(GOLD, "reference_small.pt"))["add_additional_channels"]
    assert torch.equal(gold["w"], w) and gold["num_additional_channels"] == 5
    assert torch.equal(gold["out"], mine["input_blocks.0.0.weight"])
    # the widened tiny model loads into the inpainting variant
    from ldm.util import instantiate_from_config
    sd = synthetic_state_dict(NAMED_CONFIGS["tiny"], 0)
    CK.add_additional_channels(sd, 5)
    m = instantiate_from_config(model_config(NAMED_CONFIGS["tiny_inpaint"]))
    m.load_state_dict(sd)
    assert m.input_blocks[0][0].weight.shape[1] == 9
