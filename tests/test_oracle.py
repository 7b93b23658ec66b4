"""CPU: the oracle (oracle/streaming_svd_oracle.py) reproduces the golden vectors that oracle/make_golden.py
recorded from the UNMODIFIED reference modules (tests/golden/*.npz), and the parameter grammar is stable."""
import dataclasses
import os

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("name", ["tiny_t8_16x16", "tiny_apm_t8_16x16", "tiny_t25_8x16", "tiny_t7_24x40"])
def test_oracle_matches_reference_golden(name):
    from oracle import streaming_svd_oracle as orc
    from streamingt2v_b200 import arch, synth
    g = np.load(os.path.join(GOLDEN, f"streaming_{name}.npz"))
    T, h, w, ctx_tokens, seed, use_apm, mc = (int(v) for v in g["meta"])
    cstep = int(g["ctrl_cstep"][0]) if "ctrl_cstep" in g else 1      # channels kept of the ControlNet taps
    cfg = dataclasses.replace(arch.TINY, use_apm=bool(use_apm))
    assert cfg.model_channels == mc
    sd_u = arch.synth_state_dict(arch.unet_param_shapes(cfg), seed=seed)
    sd_c = arch.synth_state_dict(arch.controlnet_param_shapes(cfg), seed=seed + 1000)
    x, t, c, kw = synth.make_inputs(cfg, T=T, h=h, w=w, seed=seed, ctx_tokens=ctx_tokens)
    taps = {}
    with torch.no_grad():
        out = orc.streaming_wrapper_forward(sd_u, sd_c, cfg, x, t, c, taps=taps, **kw)
    ref = torch.from_numpy(g["out"])
    assert out.shape == ref.shape
    assert (out - ref).abs().max().item() <= 2e-4 * max(1.0, ref.abs().max().item())
    assert (taps["ctrl.middle"][:, ::cstep] - torch.from_numpy(g["ctrl_mid"])).abs().max().item() <= 1e-3
    assert (taps["ctrl.input_blocks.11"][:, ::cstep] - torch.from_numpy(g["ctrl_hs_last"])).abs().max().item() <= 1e-3
    # the generator itself recorded |oracle - reference| at generation time
    assert float(g["oracle_vs_reference_maxerr"][0]) < 1e-4


def test_grammar_counts():
    """Tensor / parameter counts of the full-size grammar (pinned against the reference's state_dict() by
    oracle/make_golden.py for the reduced config; SURVEY.md App. A gives the full-size totals)."""
    from streamingt2v_b200 import arch
    cfg = arch.UNetConfig()
    u = arch.unet_param_shapes(cfg)
    c = arch.controlnet_param_shapes(cfg)
    nu = sum(int(np.prod(s)) for s in u.values())
    nc = sum(int(np.prod(s)) for s in c.values())
    assert len(u) == 1571 and len(c) == 657
    assert abs(nu / 1e6 - 1593.5) < 0.1 and abs(nc / 1e6 - 673.0) < 0.1


@pytest.mark.parametrize("name", ["vae_enc_2_64x96", "vae_enc_1_128x64"])
def test_vae_encoder_oracle_matches_reference_golden(name):
    """oracle/vae_encoder_oracle.py against the outputs of the unmodified reference Encoder (+ quant_conv, mode)."""
    import os

    import numpy as np
    import torch
    from oracle import vae_encoder_oracle as eorc
    from oracle.make_golden_vae_enc import make_image
    from streamingt2v_b200 import arch
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", f"{name}.npz"))
    n, H, W, seed = (int(v) for v in g["meta"])
    cfg = arch.VaeConfig()
    sd = arch.synth_state_dict(arch.vae_encoder_param_shapes(cfg), seed=seed)
    with torch.no_grad():
        out = eorc.encode(sd, cfg, make_image(n, H, W, seed))
    ref = torch.from_numpy(g["out"])
    assert (out - ref).abs().max().item() <= 2e-4 * max(1.0, ref.abs().max().item())
