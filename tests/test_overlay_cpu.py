"""The documented drop-in recipe (INTEGRATION.md 1): this repo FIRST on sys.path, the reference checkout after it.
The hot-path modules must resolve to this repo, everything else of the reference must stay importable
(ldm.models.autoencoder is what gligen_inference.load_ckpt instantiates next to the UNet, gligen_inference.py:70-86),
and names the drop-in modules do not define must fall through to the reference (gligen_b200/_overlay.py)."""
import os
import subprocess
import sys
import textwrap
import zipfile

import pytest
import torch

from conftest import GOLD, ROOT
from oracle import build_ref
from oracle.ref_harness import REF_DIR as REF

SCRIPT = textwrap.dedent('''
    import sys
    sys.path[:0] = [%(repo)r, %(ref)r]
    import ldm
    assert ldm.__path__[0].startswith(%(repo)r) and any(p.startswith(%(ref)r) for p in ldm.__path__), ldm.__path__
    # what load_ckpt needs: autoencoder (reference), UNetModel / samplers / diffusion / adapters (this repo)
    from ldm.models.autoencoder import AutoencoderKL
    import ldm.modules.diffusionmodules.model as M
    assert M.__file__.startswith(%(ref)r), M.__file__
    from ldm.util import instantiate_from_config
    U = instantiate_from_config.__globals__["get_obj_from_str"]("ldm.modules.diffusionmodules.openaimodel.UNetModel")
    assert sys.modules[U.__module__].__file__.startswith(%(repo)r)
    for dotted in ("ldm.models.diffusion.plms.PLMSSampler", "ldm.models.diffusion.ddim.DDIMSampler",
                   "ldm.models.diffusion.ldm.LatentDiffusion", "grounding_input.text_grounding_tokinzer_input.GroundingNetInput",
                   "ldm.modules.diffusionmodules.text_grounding_net.PositionNet"):
        c = instantiate_from_config.__globals__["get_obj_from_str"](dotted)
        assert sys.modules[c.__module__].__file__.startswith(%(repo)r), dotted
    from ldm.modules.attention import GatedCrossAttentionDense, GatedSelfAttentionDense, LinearAttention     # set_alpha_scale's import
    assert LinearAttention.__module__ == "ldm.modules.attention"
    # names only the reference defines fall through
    from ldm.modules.attention import GEGLU
    from ldm.modules.diffusionmodules.util import checkpoint, conv_nd, zero_module
    from ldm.util import log_txt_as_img
    assert "_gligen_b200_shadowed" in GEGLU.__module__ and "_gligen_b200_shadowed" in conv_nd.__module__
    import grounding_input.hed_grounding_tokinzer_input as H            # spatial modalities are drop-ins too since round 2
    assert H.__file__.startswith(%(repo)r)
    import ldm.modules.diffusionmodules.hed_grounding_net as HN, ldm.modules.diffusionmodules.sem_grounding_downsampler as SD
    assert HN.__file__.startswith(%(repo)r) and SD.__file__.startswith(%(repo)r)
    E = instantiate_from_config.__globals__["get_obj_from_str"]("ldm.modules.encoders.modules.FrozenCLIPEmbedder")     # config['text_encoder']
    assert sys.modules[E.__module__].__file__.startswith(%(repo)r)
    import ldm.modules.diffusionmodules.grounding_net_example as EX       # a reference-only module next to them still resolves
    assert EX.__file__.startswith(%(ref)r)
    # the reference VAE decoder actually runs in this overlay (tiny config)
    import torch
    dd = dict(double_z=True, z_channels=4, resolution=32, in_channels=3, out_ch=3, ch=32, ch_mult=[1, 2], num_res_blocks=1,
              attn_resolutions=[], dropout=0.0)
    vae = AutoencoderKL(ddconfig=dd, embed_dim=4, scale_factor=0.18215).eval()
    with torch.no_grad():
        img = vae.decode(torch.randn(1, 4, 16, 16))
    assert img.shape == (1, 3, 32, 32)
    # own LinearAttention == the reference's on the same weights
    R = sys.modules["_gligen_b200_shadowed.ldm.modules.attention"].LinearAttention
    torch.manual_seed(0)
    a, b = LinearAttention(32), R(32)
    b.load_state_dict(a.state_dict())
    x = torch.randn(2, 32, 8, 8)
    assert (a(x) - b(x)).abs().max().item() < 1e-5
    print("overlay ok")
''')


def _reference_checkout(tmp_path):
    """The reference tree to overlay: the archive build() makes (oracle/_ref) unpacked into tmp_path, else a checkout."""
    if build_ref.available():
        d = tmp_path / "reference"
        with zipfile.ZipFile(build_ref.ZIP) as z:
            z.extractall(d)
        return str(d)
    if os.path.isdir(REF):
        return REF
    pytest.skip("neither oracle/_ref (made by build() from a reference checkout) nor a reference checkout is present")


def test_repo_overlays_reference_checkout(tmp_path):
    ref = _reference_checkout(tmp_path)
    r = subprocess.run([sys.executable, "-c", SCRIPT % dict(repo=ROOT, ref=ref)], cwd=str(tmp_path), capture_output=True, text=True,
                       env={k: v for k, v in os.environ.items() if k != "PYTHONPATH"})
    assert r.returncode == 0 and "overlay ok" in r.stdout, r.stdout + r.stderr


def test_repo_alone_reports_missing_reference_names(tmp_path):
    """Without a reference checkout behind it, a name the drop-in does not define is an ordinary AttributeError."""
    code = textwrap.dedent('''
        import sys
        sys.path.insert(0, %r)
        import ldm.modules.attention as A
        assert hasattr(A, "GatedSelfAttentionDense") and hasattr(A, "LinearAttention")
        try:
            A.GEGLU
        except AttributeError as e:
            assert "no reference checkout" in str(e)
            print("ok")
    ''') % ROOT
    env = {k: v for k, v in os.environ.items() if k != "PYTHONPATH"}
    r = subprocess.run([sys.executable, "-c", code], cwd=str(tmp_path), capture_output=True, text=True, env=env)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def test_repo_overlays_stub_checkout(tmp_path):
    """The overlay mechanics without the reference: a stub checkout (namespace `ldm`, one name per shadowed module and a
    module of its own) behind this repo.  Drop-in modules win, the stub's own module imports, names only it defines fall
    through, and its shadowed modules are loaded under the private alias."""
    stub = tmp_path / "checkout"
    files = {"ldm/modules/attention.py": "class GEGLU:\n    pass\n",
             "ldm/modules/diffusionmodules/util.py": "def conv_nd(*a):\n    return 'stub conv_nd'\n",
             "ldm/modules/diffusionmodules/grounding_net_example.py": "WHO = 'stub'\n",
             "ldm/util.py": "def log_txt_as_img(*a):\n    return 'stub log'\n"}
    for rel, text in files.items():
        (stub / rel).parent.mkdir(parents=True, exist_ok=True)
        (stub / rel).write_text(text)
    code = textwrap.dedent('''
        import sys
        sys.path[:0] = [%(repo)r, %(ref)r]
        import ldm
        assert ldm.__path__[0].startswith(%(repo)r) and any(p.startswith(%(ref)r) for p in ldm.__path__), ldm.__path__
        from ldm.modules.attention import GatedSelfAttentionDense, GEGLU, LinearAttention
        assert sys.modules[GatedSelfAttentionDense.__module__].__file__.startswith(%(repo)r)
        assert LinearAttention.__module__ == "ldm.modules.attention" and "_gligen_b200_shadowed" in GEGLU.__module__
        from ldm.modules.diffusionmodules.util import conv_nd
        from ldm.util import instantiate_from_config, log_txt_as_img
        assert conv_nd() == "stub conv_nd" and log_txt_as_img() == "stub log"
        import ldm.modules.diffusionmodules.grounding_net_example as EX
        assert EX.__file__.startswith(%(ref)r) and EX.WHO == "stub"
        U = instantiate_from_config.__globals__["get_obj_from_str"]("ldm.modules.diffusionmodules.openaimodel.UNetModel")
        assert sys.modules[U.__module__].__file__.startswith(%(repo)r)
        import ldm.modules.attention as A
        try:
            A.NOT_IN_EITHER
        except AttributeError as e:
            assert "no reference checkout" not in str(e)
            print("ok")
    ''') % dict(repo=ROOT, ref=str(stub))
    env = {k: v for k, v in os.environ.items() if k != "PYTHONPATH"}
    r = subprocess.run([sys.executable, "-c", code], cwd=str(tmp_path), capture_output=True, text=True, env=env)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


@torch.no_grad()
def test_linear_attention_matches_reference():
    """The drop-in LinearAttention against the reference's output on the same weights and input
    (tests/golden/reference_small.pt, oracle/gen_golden_small.py)."""
    from ldm.modules.attention import LinearAttention
    gold = torch.load(os.path.join(GOLD, "reference_small.pt"))["linear_attention"]
    la = LinearAttention(gold["dim"]).eval()
    la.load_state_dict(gold["state_dict"])
    assert (la(gold["x"]) - gold["out"]).abs().max().item() < 1e-5
