"""Pin the oracle against the REAL reference and write tests/golden/*.pt.   (run in the authoring
container only; /root/reference does not exist on the GPU box)

    python oracle/gen_golden.py [--full] [--tiny]

For each configuration it
  1. builds the unmodified reference `UNetModel` (imported from /root/reference), loads the seeded
     synthetic weights (gligen_b200.spec.synthetic_state_dict) with strict key checking,
  2. runs reference forwards / reference PLMSSampler / DDIMSampler on seeded synthetic inputs,
  3. asserts the oracle restatement (oracle/unet_oracle.py, oracle/sampler_oracle.py) agrees to fp32
     round-off, and
  4. stores the REFERENCE outputs as golden fixtures.
"""
from __future__ import annotations

import argparse
import hashlib
import os
import sys
import time
from functools import partial

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
sys.path.insert(0, REF)      # reference `grounding_input`, `inpaint_mask_func`, ... win over the repo's drop-in modules
sys.path.insert(1, REPO)


def _mount_reference_package(name: str) -> None:
    """The reference's `ldm` is a namespace package (no __init__.py) while the repo's drop-in `ldm` is a regular one,
    which would win the import whatever the sys.path order: register `ldm` with the reference directory as its only
    search location so that every `ldm.*` import below executes REFERENCE code."""
    import importlib.machinery
    import types
    path = os.path.join(REF, name)
    spec = importlib.machinery.ModuleSpec(name, None, is_package=True)
    spec.submodule_search_locations = [path]
    mod = types.ModuleType(name)
    mod.__path__ = [path]
    mod.__spec__ = spec
    sys.modules[name] = mod


_mount_reference_package("ldm")

from gligen_b200.spec import NAMED_CONFIGS, synthetic_state_dict  # noqa: E402
from gligen_b200 import synth  # noqa: E402
from oracle import unet_oracle as UO  # noqa: E402
from oracle import sampler_oracle as SO  # noqa: E402

GOLD = os.path.join(REPO, "tests", "golden")


def ref_model(cfg):
    from ldm.modules.diffusionmodules.openaimodel import UNetModel
    assert UNetModel.__module__ and "/root/reference" in sys.modules[UNetModel.__module__].__file__
    tok = {
        "text": ("ldm.modules.diffusionmodules.text_grounding_net.PositionNet", dict(in_dim=cfg.tok_in_dim, out_dim=cfg.tok_out_dim)),
        "text_image": ("ldm.modules.diffusionmodules.text_image_grounding_net.PositionNet", dict(in_dim=cfg.tok_in_dim, out_dim=cfg.tok_out_dim)),
        "keypoint": ("ldm.modules.diffusionmodules.keypoint_grounding_net.PositionNet", dict(max_persons_per_image=cfg.max_persons, out_dim=cfg.tok_out_dim)),
    }[cfg.tokenizer]
    m = UNetModel(image_size=cfg.image_size, in_channels=cfg.in_channels, out_channels=cfg.out_channels,
                  model_channels=cfg.model_channels, attention_resolutions=list(cfg.attention_resolutions),
                  num_res_blocks=cfg.num_res_blocks, channel_mult=list(cfg.channel_mult), num_heads=cfg.num_heads,
                  transformer_depth=1, context_dim=cfg.context_dim, fuser_type="gatedSA", use_checkpoint=True,
                  inpaint_mode=cfg.inpaint_mode, grounding_tokenizer=dict(target=tok[0], params=tok[1]))
    return m.eval()


def ref_grounding_input(cfg):
    import importlib
    name = {"text": "text_grounding_tokinzer_input", "text_image": "text_image_grounding_tokinzer_input",
            "keypoint": "keypoint_grounding_tokinzer_input"}[cfg.tokenizer]
    return importlib.import_module(f"grounding_input.{name}").GroundingNetInput()


def set_alpha_scale(model, alpha_scale):
    """gligen_inference.py:24-28 (gligen_inference.py itself cannot be imported here: needs clip/omegaconf)."""
    from ldm.modules.attention import GatedCrossAttentionDense, GatedSelfAttentionDense
    for module in model.modules():
        if type(module) == GatedCrossAttentionDense or type(module) == GatedSelfAttentionDense:
            module.scale = alpha_scale


def check(name, a, b, tol):
    err = (a - b).abs().max().item()
    ref = b.abs().max().item()
    print(f"    {name}: max|oracle-ref| = {err:.3e} (ref max {ref:.3f})")
    assert err <= tol * max(1.0, ref), (name, err)


@torch.no_grad()
def run_config(name, B, max_objs, plms_S, alpha_type, ddim_S, n_valid=None, do_sampling=True):
    cfg = NAMED_CONFIGS[name]
    print(f"== {name}: B={B} max_objs={max_objs}")
    t0 = time.time()
    sd = synthetic_state_dict(cfg, seed=0)
    model = ref_model(cfg)
    missing = model.load_state_dict(sd, strict=True)
    print(f"   weights+model {time.time()-t0:.1f}s  {missing}")
    gin = ref_grounding_input(cfg)
    model.grounding_tokenizer_input = gin
    inp = synth.make_inputs(cfg, B, max_objs, seed=2, n_valid=n_valid)
    grounding = gin.prepare(inp["batch"])
    for k, v in synth.grounding_kwargs(cfg, inp["batch"]).items():
        assert torch.equal(v, grounding[k]), k
    extra = None
    mask = z0 = None
    if cfg.inpaint_mode:
        from inpaint_mask_func import draw_masks_from_boxes
        mask = draw_masks_from_boxes(inp["batch"]["boxes"], cfg.image_size)
        assert torch.equal(mask, SO.draw_masks_from_boxes(inp["batch"]["boxes"], cfg.image_size))
        z0 = inp["z0"]
        extra = torch.cat([z0 * mask, mask], dim=1)

    out = {"cfg": name, "B": B, "max_objs": max_objs, "n_valid": n_valid}
    # ---- single forwards: cond / null, scale 1 and 0.5 and 0 ------------------------------
    ts = torch.tensor([981, 501, 21, 1][:B] if B <= 4 else [981] * B, dtype=torch.long)
    fw = {}
    for scale in (1.0, 0.5, 0.0):
        set_alpha_scale(model, scale)
        t1 = time.time()
        e_c = model(dict(x=inp["x"], timesteps=ts, context=inp["context"], grounding_input=grounding,
                         inpainting_extra_input=extra, grounding_extra_input=None))
        e_u = model(dict(x=inp["x"], timesteps=ts, context=inp["uc"],
                         inpainting_extra_input=extra, grounding_extra_input=None))
        print(f"   ref forwards scale={scale}: {time.time()-t1:.1f}s  eps std {e_c.std():.3f} max {e_c.abs().max():.3f}")
        o_c = UO.unet_forward(cfg, sd, inp["x"], ts, inp["context"], grounding, scale, extra)
        o_u = UO.unet_forward(cfg, sd, inp["x"], ts, inp["uc"], UO.null_grounding(cfg, grounding), scale, extra)
        check(f"eps_cond s={scale}", o_c, e_c, 2e-4)
        check(f"eps_null s={scale}", o_u, e_u, 2e-4)
        fw[scale] = {"eps_cond": e_c.clone(), "eps_null": e_u.clone()}
    out["timesteps"] = ts
    out["forward"] = fw

    # ---- sampling loops through the reference sampler classes ----------------------------
    if do_sampling:
        from ldm.models.diffusion.plms import PLMSSampler
        from ldm.models.diffusion.ddim import DDIMSampler
        from ldm.models.diffusion.ldm import LatentDiffusion
        diffusion = LatentDiffusion(linear_start=0.00085, linear_end=0.012, timesteps=1000)
        sched = SO.make_schedule()
        for k in ("betas", "alphas_cumprod", "alphas_cumprod_prev", "sqrt_alphas_cumprod", "sqrt_one_minus_alphas_cumprod"):
            assert torch.equal(getattr(diffusion, k), sched[k]), k
        shape = (B, cfg.in_channels, cfg.image_size, cfg.image_size)
        sd_conv = torch.load(os.path.join(REF, "SD_input_conv_weight_bias.pth"))

        def sample(kind, S, atype, guidance):
            cls = PLMSSampler if kind == "plms" else DDIMSampler
            m = ref_model(cfg)                     # fresh: restore_first_conv_from_SD mutates the model
            m.load_state_dict(sd, strict=True)
            m.grounding_tokenizer_input = gin
            sampler = cls(diffusion, m, alpha_generator_func=partial(SO.alpha_generator, type=atype),
                          set_alpha_scale=set_alpha_scale)
            input = dict(x=inp["x"].clone(), timesteps=None, context=inp["context"], grounding_input=grounding,
                         inpainting_extra_input=extra, grounding_extra_input=None)
            torch.manual_seed(1234)
            t1 = time.time()
            ref = sampler.sample(S=S, shape=shape, input=input, uc=inp["uc"], guidance_scale=guidance, mask=mask, x0=z0)
            print(f"   ref {kind} S={S} alpha={atype}: {time.time()-t1:.1f}s  latent std {ref.std():.3f}")
            # oracle twin
            state = {"scale": 1.0, "sd": dict(sd)}

            def on_alpha(a):
                state["scale"] = a
                if a == 0 and not cfg.inpaint_mode:          # openaimodel.py:400-413
                    state["sd"]["input_blocks.0.0.weight"] = sd_conv["weight"]
                    state["sd"]["input_blocks.0.0.bias"] = sd_conv["bias"]

            def eps_fn(x, t, cond):
                gr = grounding if cond else UO.null_grounding(cfg, grounding)
                ctx = inp["context"] if cond else inp["uc"]
                return UO.unet_forward(cfg, state["sd"], x, t, ctx, gr, state["scale"], extra)

            fn = SO.plms_sample if kind == "plms" else SO.ddim_sample
            torch.manual_seed(1234)
            got = fn(eps_fn, S, shape, sched, x_T=inp["x"].clone(), use_cfg=True, guidance_scale=guidance,
                     alphas=SO.alpha_generator(S, atype), on_alpha=on_alpha, mask=mask, x0=z0)
            check(f"{kind} S={S}", got, ref, 5e-4)
            return ref.clone()

        cwd = os.getcwd()
        os.chdir(REF)                                  # restore_first_conv_from_SD uses a CWD-relative path
        try:
            restorable = (not cfg.inpaint_mode) and cfg.model_channels == 320
            atype = alpha_type if (restorable or cfg.inpaint_mode) else [1, 0, 0]
            out["plms"] = {"S": plms_S, "alpha_type": atype, "guidance": 7.5, "latent": sample("plms", plms_S, atype, 7.5)}
            out["ddim"] = {"S": ddim_S, "alpha_type": [1, 0, 0], "guidance": 7.5, "latent": sample("ddim", ddim_S, [1, 0, 0], 7.5)}
        finally:
            os.chdir(cwd)
    os.makedirs(GOLD, exist_ok=True)
    path = os.path.join(GOLD, f"{name}_B{B}_G{max_objs}.pt")
    torch.save(out, path)
    print(f"   wrote {path} ({os.path.getsize(path)/1024:.0f} KiB)")


@torch.no_grad()
def run_plms50(name="sd14_box_text", B=1, max_objs=30, S=50, alpha_types=((1, 0, 0), (0.3, 0, 0.7)), twin_for=((0.3, 0, 0.7),)):
    """The path the metric is quoted on: reference PLMSSampler.sample(S=50, guidance 7.5) at full size (102 UNet
    forwards), for alpha_type [1,0,0] and the script default [0.3,0,0.7] (gligen_inference.py:389-390,475).
    Stores the REFERENCE fp32 final latents; the oracle twin is re-checked on `twin_for`."""
    cfg = NAMED_CONFIGS[name]
    sd = synthetic_state_dict(cfg, seed=0)
    gin = ref_grounding_input(cfg)
    inp = synth.make_inputs(cfg, B, max_objs, seed=2)
    grounding = gin.prepare(inp["batch"])
    from ldm.models.diffusion.plms import PLMSSampler
    from ldm.models.diffusion.ldm import LatentDiffusion
    diffusion = LatentDiffusion(linear_start=0.00085, linear_end=0.012, timesteps=1000)
    sched = SO.make_schedule()
    shape = (B, cfg.in_channels, cfg.image_size, cfg.image_size)
    sd_conv = torch.load(os.path.join(REF, "SD_input_conv_weight_bias.pth"))
    out = {"cfg": name, "B": B, "max_objs": max_objs, "n_valid": None, "S": S, "guidance": 7.5, "runs": {}}
    cwd = os.getcwd()
    os.chdir(REF)
    try:
        for atype in alpha_types:
            atype = list(atype)
            m = ref_model(cfg)
            m.load_state_dict(sd, strict=True)
            m.grounding_tokenizer_input = gin
            sampler = PLMSSampler(diffusion, m, alpha_generator_func=partial(SO.alpha_generator, type=atype), set_alpha_scale=set_alpha_scale)
            input = dict(x=inp["x"].clone(), timesteps=None, context=inp["context"], grounding_input=grounding,
                         inpainting_extra_input=None, grounding_extra_input=None)
            torch.manual_seed(1234)
            t1 = time.time()
            ref = sampler.sample(S=S, shape=shape, input=input, uc=inp["uc"], guidance_scale=7.5)
            print(f"   ref plms S={S} alpha={atype}: {time.time()-t1:.1f}s  latent std {ref.std():.3f} max {ref.abs().max():.3f}", flush=True)
            del m, sampler
            twin = None
            if tuple(atype) in [tuple(t) for t in twin_for]:
                state = {"scale": 1.0, "sd": dict(sd)}

                def on_alpha(a):
                    state["scale"] = a
                    if a == 0:
                        state["sd"]["input_blocks.0.0.weight"] = sd_conv["weight"]
                        state["sd"]["input_blocks.0.0.bias"] = sd_conv["bias"]

                def eps_fn(x, t, cond):
                    gr = grounding if cond else UO.null_grounding(cfg, grounding)
                    return UO.unet_forward(cfg, state["sd"], x, t, inp["context"] if cond else inp["uc"], gr, state["scale"], None)

                torch.manual_seed(1234)
                got = SO.plms_sample(eps_fn, S, shape, sched, x_T=inp["x"].clone(), use_cfg=True, guidance_scale=7.5,
                                     alphas=SO.alpha_generator(S, atype), on_alpha=on_alpha)
                check(f"plms S={S} alpha={atype} oracle twin", got, ref, 5e-4)
                twin = (got - ref).abs().max().item()
            out["runs"][str(atype)] = {"alpha_type": atype, "latent": ref.clone(), "oracle_twin_max_abs": twin}
            torch.save(out, os.path.join(GOLD, f"{name}_B{B}_G{max_objs}_plms{S}.pt"))        # keep partial results
    finally:
        os.chdir(cwd)
    print(f"   wrote {name}_B{B}_G{max_objs}_plms{S}.pt")


def scalar_anchors():
    """Closed-form anchors from SURVEY 8c, checked against reference code and stored."""
    from ldm.modules.diffusionmodules.util import timestep_embedding, FourierEmbedder
    te = timestep_embedding(torch.tensor([981, 1]), 320)
    assert torch.allclose(te, UO.timestep_embedding(torch.tensor([981, 1]), 320), atol=1e-6)
    box = torch.tensor([[0.25, 0.5, 0.75, 1.0]])
    fe = FourierEmbedder(num_freqs=8)(box)
    assert torch.allclose(fe, UO.fourier_embed(box, 8), atol=1e-6)
    sched = SO.make_schedule()
    steps = SO.ddim_timesteps(50)
    sig, al, alp = SO.ddim_parameters(sched["alphas_cumprod"], steps)
    torch.save({"timestep_embedding_981_1": te, "fourier_box": fe, "alphas_cumprod": sched["alphas_cumprod"],
                "ddim50_alphas": torch.tensor(al), "ddim50_alphas_prev": torch.tensor(alp)},
               os.path.join(GOLD, "scalar_anchors.pt"))
    print("anchors:", te[0, :2].tolist(), fe[0, :4].tolist(), float(sched["alphas_cumprod"][0]), float(al[0]), float(al[-1]), float(alp[-1]))


def run_vae(name, B, seed=3, store_half=False, image_stride=1):
    """SURVEY 8(f) rank 1 (next row): pin oracle/vae_oracle.py against the reference AutoencoderKL.decode."""
    from gligen_b200.spec import NAMED_VAE_CONFIGS, synthetic_vae_state_dict, vae_decoder_param_shapes
    from oracle import vae_oracle as VO
    from ldm.models.autoencoder import AutoencoderKL
    assert "/root/reference" in sys.modules[AutoencoderKL.__module__].__file__
    cfg = NAMED_VAE_CONFIGS[name]
    dd = dict(double_z=True, z_channels=cfg.z_channels, resolution=cfg.image_size, in_channels=3, out_ch=cfg.out_ch, ch=cfg.ch,
              ch_mult=list(cfg.ch_mult), num_res_blocks=cfg.num_res_blocks, attn_resolutions=[], dropout=0.0)
    ref = AutoencoderKL(ddconfig=dd, embed_dim=cfg.embed_dim, scale_factor=cfg.scale_factor).eval()
    ref_keys = [(k, tuple(v.shape)) for k, v in ref.state_dict().items() if k.startswith(("decoder.", "post_quant_conv."))]
    mine = [(k, tuple(s)) for k, s in vae_decoder_param_shapes(cfg).items()]
    assert sorted(ref_keys) == sorted(mine), "decoder state-dict keys / shapes differ from the reference"
    assert [k for k, _ in ref_keys if k.startswith("decoder.")] == [k for k, _ in mine if k.startswith("decoder.")], "registration order differs"
    sd = synthetic_vae_state_dict(cfg, 0)
    missing, unexpected = ref.load_state_dict(sd, strict=False)
    assert not unexpected and all(k.startswith(("encoder.", "quant_conv.")) for k in missing)
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(B, cfg.embed_dim, cfg.latent_size, cfg.latent_size, generator=g) * cfg.scale_factor * 4.0   # latents ~ 0.18215 * N(0, ~4^2)
    t0 = time.time()
    with torch.no_grad():
        img = ref.decode(z)
    t_ref = time.time() - t0
    mine_img = VO.vae_decode(cfg, sd, z)
    diff = (img - mine_img).abs().max().item()
    print(f"{name}: reference decode {tuple(img.shape)} in {t_ref:.1f} s; max |oracle - reference| = {diff:.3e}; mean |img| = {img.abs().mean():.3f}")
    assert diff <= 1e-4 * max(1.0, img.abs().max().item())
    img = img[..., ::image_stride, ::image_stride]          # every image_stride-th row and column: keeps the fixture under 1 MB
    torch.save({"name": name, "B": B, "seed": seed, "z": z, "image": img.half() if store_half else img, "image_stride": image_stride,
                "oracle_max_abs_diff": diff},
               os.path.join(GOLD, f"{name}_B{B}.pt"))


def run_vae_encode(name, B, seed=5, store_half=False, x_from_seed=False):
    """SURVEY 8(f) rank 3 (encoder half): pin oracle/vae_oracle.vae_encode_moments / vae_encode against the reference
    AutoencoderKL.encode (same synthetic weights, same image, same global CPU seed for the posterior noise)."""
    from gligen_b200.spec import NAMED_VAE_CONFIGS, synthetic_vae_encoder_state_dict, vae_encoder_param_shapes
    from oracle import vae_oracle as VO
    from ldm.models.autoencoder import AutoencoderKL
    assert "/root/reference" in sys.modules[AutoencoderKL.__module__].__file__
    cfg = NAMED_VAE_CONFIGS[name]
    dd = dict(double_z=True, z_channels=cfg.z_channels, resolution=cfg.image_size, in_channels=cfg.in_channels, out_ch=cfg.out_ch, ch=cfg.ch,
              ch_mult=list(cfg.ch_mult), num_res_blocks=cfg.num_res_blocks, attn_resolutions=[], dropout=0.0)
    ref = AutoencoderKL(ddconfig=dd, embed_dim=cfg.embed_dim, scale_factor=cfg.scale_factor).eval()
    ref_keys = [(k, tuple(v.shape)) for k, v in ref.state_dict().items() if k.startswith(("encoder.", "quant_conv."))]
    mine = [(k, tuple(s)) for k, s in vae_encoder_param_shapes(cfg).items()]
    assert ref_keys == mine, "encoder state-dict keys / shapes / registration order differ from the reference"
    sd = synthetic_vae_encoder_state_dict(cfg, 1)
    missing, unexpected = ref.load_state_dict(sd, strict=False)
    assert not unexpected and all(k.startswith(("decoder.", "post_quant_conv.")) for k in missing)
    x = VO.encode_test_image(cfg, B, seed)
    if store_half:
        x = x.half().float()               # the fixture stores the image as fp16: run the reference on exactly those values
    t0 = time.time()
    with torch.no_grad():
        mom = ref.quant_conv(ref.encoder(x))
        torch.manual_seed(1234)
        z0 = ref.encode(x)
    t_ref = time.time() - t0
    mine_mom = VO.vae_encode_moments(cfg, sd, x)
    torch.manual_seed(1234)
    mine_z0 = VO.vae_encode(cfg, sd, x)
    diff = (mom - mine_mom).abs().max().item()
    diff_z = (z0 - mine_z0).abs().max().item()
    print(f"{name}: reference encode {tuple(x.shape)} -> {tuple(mom.shape)} in {t_ref:.1f} s; max |oracle - reference| moments {diff:.3e}, "
          f"sample {diff_z:.3e}; mean |mean| {mom[:, :cfg.embed_dim].abs().mean():.3f}, logvar range [{mom[:, cfg.embed_dim:].min():.2f}, {mom[:, cfg.embed_dim:].max():.2f}]")
    assert diff <= 1e-4 * max(1.0, mom.abs().max().item()) and diff_z <= 1e-4 * max(1.0, z0.abs().max().item())
    out = {"name": name, "B": B, "seed": seed, "noise_seed": 1234, "moments": mom, "z0": z0, "oracle_max_abs_diff": diff}
    if x_from_seed:             # keeps the fixture under 1 MB: tests rebuild x with VO.encode_test_image and check the hash
        out["x_sha256"] = hashlib.sha256(x.half().numpy().tobytes()).hexdigest()
    else:
        out["x"] = x.half() if store_half else x
    torch.save(out, os.path.join(GOLD, f"{name}_enc_B{B}.pt"))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--full", action="store_true")
    ap.add_argument("--tiny", action="store_true")
    ap.add_argument("--vae", action="store_true", help="only the VAE-decoder fixtures (next row, SURVEY 8f)")
    ap.add_argument("--vae-enc", action="store_true", help="only the VAE-encoder fixtures (SURVEY 8f rank 3, encoder half)")
    ap.add_argument("--configs345", action="store_true", help="full-size single forwards (+ short inpaint loops) for BASELINE configs 3, 4, 5")
    ap.add_argument("--plms50", action="store_true", help="50-step PLMS + CFG final latents at full size (the path the metric is quoted on)")
    args = ap.parse_args()
    torch.set_num_threads(os.cpu_count())
    os.makedirs(GOLD, exist_ok=True)
    if args.vae:
        run_vae("tiny_vae", B=2)
        run_vae("tiny_vae64", B=2)
        run_vae("small_vae", B=1, store_half=True)
        run_vae("sd14_vae", B=1, store_half=True, image_stride=2)
        sys.exit(0)
    if args.vae_enc:
        run_vae_encode("tiny_vae", B=2)
        run_vae_encode("tiny_vae64", B=2)
        run_vae_encode("small_vae", B=1, store_half=True)
        run_vae_encode("sd14_vae", B=1, store_half=True, x_from_seed=True)
        sys.exit(0)
    if args.configs345:
        # BASELINE config 3 (box + text + image: 30 objects -> 60 grounding tokens), config 5 (keypoint: 8 x 17 = 136
        # tokens), config 4 (inpainting: 9-channel first conv, scheduled sampling [0.3,0,0.7], per-step blend)
        run_config("sd14_box_text_image", B=1, max_objs=30, plms_S=0, alpha_type=[1, 0, 0], ddim_S=0, do_sampling=False)
        run_config("sd14_keypoint", B=1, max_objs=136, plms_S=0, alpha_type=[1, 0, 0], ddim_S=0, do_sampling=False)
        run_config("sd14_inpaint_box_text", B=1, max_objs=30, plms_S=4, alpha_type=[0.3, 0, 0.7], ddim_S=2)
    if args.plms50:
        run_plms50()
    if args.configs345 or args.plms50:
        sys.exit(0)
    if args.tiny or not args.full:
        scalar_anchors()
        run_config("tiny", B=2, max_objs=6, plms_S=4, alpha_type=[0.5, 0, 0.5], ddim_S=2)
        run_config("tiny_text_image", B=2, max_objs=5, plms_S=4, alpha_type=[1, 0, 0], ddim_S=2)
        run_config("tiny_keypoint", B=2, max_objs=34, plms_S=4, alpha_type=[1, 0, 0], ddim_S=2)
        run_config("tiny_inpaint", B=2, max_objs=6, plms_S=4, alpha_type=[0.5, 0, 0.5], ddim_S=2)
    if args.full:
        # the SD first conv (real SD-1.4 weights bundled with the reference) is needed by the
        # restore_first_conv_from_SD step on the GPU box: keep a copy as a data fixture.
        w = torch.load(os.path.join(REF, "SD_input_conv_weight_bias.pth"))
        torch.save({"weight": w["weight"].clone(), "bias": w["bias"].clone()}, os.path.join(GOLD, "SD_input_conv_weight_bias.pth"))
        # BASELINE config 1: 1x4x64x64, 2 DDIM steps, 2 box+text tokens; plus PLMS S=4 with the
        # scheduled-sampling first-conv swap, and B=1 single forwards at G=30.
        run_config("sd14_box_text", B=1, max_objs=2, plms_S=4, alpha_type=[0.5, 0, 0.5], ddim_S=2, n_valid=2)
        run_config("sd14_box_text", B=1, max_objs=30, plms_S=0, alpha_type=[1, 0, 0], ddim_S=0, do_sampling=False)
