"""Run two small pieces of the UNMODIFIED reference and write what they return to tests/golden/reference_small.pt
(needs the reference checkout, oracle/ref_harness.REF_DIR).

  * convert_ckpt.add_additional_channels(sd, 5) on a seeded 320-channel first conv (tests/test_checkpoint_cpu.py);
  * ldm.modules.attention.LinearAttention(32) on seeded weights and input (tests/test_overlay_cpu.py).

    python oracle/gen_golden_small.py
"""
from __future__ import annotations

import importlib.util
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import ref_harness as RH  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "reference_small.pt")


@torch.no_grad()
def main():
    RH.mount("dir")
    spec = importlib.util.spec_from_file_location("_ref_convert_ckpt", os.path.join(RH.REF_DIR, "convert_ckpt.py"))
    conv = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(conv)
    w = torch.randn(320, 4, 3, 3, generator=torch.Generator().manual_seed(0))
    sd = {"input_blocks.0.0.weight": w.clone(), "other": torch.ones(2)}
    conv.add_additional_channels(sd, 5)

    from ldm.modules.attention import LinearAttention
    assert RH.is_reference_module(LinearAttention)
    torch.manual_seed(0)
    la = LinearAttention(32).eval()
    x = torch.randn(2, 32, 8, 8)
    out = {"add_additional_channels": {"w": w, "num_additional_channels": 5, "out": sd["input_blocks.0.0.weight"]},
           "linear_attention": {"dim": 32, "state_dict": la.state_dict(), "x": x, "out": la(x)}}
    torch.save(out, OUT)
    print(f"wrote {OUT}")


if __name__ == "__main__":
    main()
