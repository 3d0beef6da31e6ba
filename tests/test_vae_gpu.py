"""VAE decoder on the GPU through the drop-in `ldm.models.autoencoder.AutoencoderKL.decode` against the REFERENCE decode
goldens (same seeded weights and latents).  Tolerance: bf16 operands / fp32 accumulation through ~30 convolutions against an
fp32 reference: rel-L2 <= 3e-2, max-abs <= 10 % of max|image| (measured values are printed)."""
import hashlib
import os

import pytest
import torch

from conftest import GOLD, assert_close
from gligen_b200.spec import NAMED_VAE_CONFIGS, synthetic_vae_encoder_state_dict, synthetic_vae_state_dict

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name,B", [("tiny_vae64", 2), ("small_vae", 1), ("sd14_vae", 1)])
def test_vae_decode_matches_reference(name, B):
    from ldm.models.autoencoder import AutoencoderKL
    cfg = NAMED_VAE_CONFIGS[name]
    gold = torch.load(os.path.join(GOLD, f"{name}_B{B}.pt"))
    dd = dict(double_z=True, z_channels=cfg.z_channels, resolution=cfg.image_size, in_channels=3, out_ch=cfg.out_ch, ch=cfg.ch,
              ch_mult=list(cfg.ch_mult), num_res_blocks=cfg.num_res_blocks, attn_resolutions=[], dropout=0.0)
    m = AutoencoderKL(ddconfig=dd, embed_dim=cfg.embed_dim, scale_factor=cfg.scale_factor)
    m.load_state_dict(synthetic_vae_state_dict(cfg, 0), strict=False)
    m = m.to("cuda:0").eval()
    img = m.decode(gold["z"].to("cuda:0"))
    torch.cuda.synchronize()
    st = gold.get("image_stride", 1)          # a full-size fixture keeps every st-th row and column of the reference image
    r, mx = assert_close(img[..., ::st, ::st], gold["image"].float(), rel=3e-2, max_rel=0.10, what=f"{name} decode")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    m.decode(gold["z"].to("cuda:0"))
    e1.record()
    torch.cuda.synchronize()
    print(f"\nVAE {name} B={B}: rel_l2={r:.3e} max_rel={mx:.3e}; decode {e0.elapsed_time(e1):.2f} ms (eager launches)")


@pytest.mark.parametrize("name,B", [("tiny_vae64", 2), ("small_vae", 1), ("sd14_vae", 1)])
def test_vae_encode_matches_reference(name, B):
    """`AutoencoderKL.encode` (inpainting front end, gligen_inference.py:403-404) against the REFERENCE moments and, with the
    same global CPU seed, the reference's posterior sample z0.  Tolerance as for decode: rel-L2 <= 3e-2, max-abs <= 10 %."""
    from ldm.models.autoencoder import AutoencoderKL
    cfg = NAMED_VAE_CONFIGS[name]
    gold = torch.load(os.path.join(GOLD, f"{name}_enc_B{B}.pt"))
    dd = dict(double_z=True, z_channels=cfg.z_channels, resolution=cfg.image_size, in_channels=3, out_ch=cfg.out_ch, ch=cfg.ch,
              ch_mult=list(cfg.ch_mult), num_res_blocks=cfg.num_res_blocks, attn_resolutions=[], dropout=0.0)
    m = AutoencoderKL(ddconfig=dd, embed_dim=cfg.embed_dim, scale_factor=cfg.scale_factor)
    sd = dict(synthetic_vae_state_dict(cfg, 0))
    sd.update(synthetic_vae_encoder_state_dict(cfg, 1))
    m.load_state_dict(sd, strict=True)
    m = m.to("cuda:0").eval()
    if "x" in gold:
        x = gold["x"].float()
    else:                                    # a full-size fixture stores the input's recipe and hash, not the image
        from oracle import vae_oracle as VO
        x = VO.encode_test_image(cfg, gold["B"], gold["seed"]).half()
        assert hashlib.sha256(x.numpy().tobytes()).hexdigest() == gold["x_sha256"]
        x = x.float()
    x = x.to("cuda:0")
    mom = m.encode_moments(x)
    torch.cuda.synchronize()
    r, mx = assert_close(mom, gold["moments"], rel=3e-2, max_rel=0.10, what=f"{name} encode moments")
    torch.manual_seed(gold["noise_seed"])
    z0 = m.encode(x)
    rz, mz = assert_close(z0, gold["z0"], rel=3e-2, max_rel=0.10, what=f"{name} encode sample")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    m.encode_moments(x)
    e1.record()
    torch.cuda.synchronize()
    print(f"\nVAE {name} B={B} encode: moments rel_l2={r:.3e} max_rel={mx:.3e}; z0 rel_l2={rz:.3e} max_rel={mz:.3e}; "
          f"{e0.elapsed_time(e1):.2f} ms (eager launches)")
