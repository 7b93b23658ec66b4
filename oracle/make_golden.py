"""ORACLE tooling — build-container only.  Generates tests/golden/*.npz from the UNMODIFIED reference modules and
pins the restatement (oracle/streaming_svd_oracle.py) and the parameter grammar (streamingt2v_b200/arch.py)
against them.

    python oracle/make_golden.py            # writes fixtures, prints max |oracle - reference|

Nothing under /root/reference is copied; the fixtures hold only output tensors (inputs and weights are re-derived
from seeds by streamingt2v_b200/{synth,arch}.py on both sides).
"""
from __future__ import annotations

import dataclasses
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_shims  # noqa: E402
from oracle import streaming_svd_oracle as orc  # noqa: E402
from streamingt2v_b200 import arch, synth  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")

CASES = {
    # name: (cfg, T, h, w, ctx_tokens, seed)
    "tiny_t8_16x16": (arch.TINY, 8, 16, 16, 1, 1),
    "tiny_t25_8x16": (arch.TINY, 25, 8, 16, 1, 2),
    "tiny_apm_t8_16x16": (dataclasses.replace(arch.TINY, use_apm=True), 8, 16, 16, 17, 3),
    # extents that are not powers of two on every level (24x40 -> 12x20 -> 6x10 -> 3x5), like the production
    # 72x128 -> 9x16: ragged 128-row tiles and TMA boxes larger than the tensor
    "tiny_t7_24x40": (arch.TINY, 7, 24, 40, 1, 4),
    # FULL network width (channel_mult (1,2,4,4): C up to 1280, 20 heads, 2560-wide concat GroupNorm, K=5120 FF2).
    # BASELINE.json configs[0]: one denoise step, 8 frames, 64x64 latent, fp32 on CPU (~50 s for the reference here)
    "full_t8_64x64": (arch.UNetConfig(), 8, 64, 64, 1, 21),
    # full width + APM (17 context tokens), 25 frames, extents that are not powers of two on any level
    "full_apm_t25_24x40": (dataclasses.replace(arch.UNetConfig(), use_apm=True), 25, 24, 40, 17, 22),
}
# every fixture stays under 1 MB: name -> (channel step of the stored ControlNet taps, latent-row step of the stored
# output); the tests slice their own tensors likewise and check the whole output against the oracle
SAMPLING = {"tiny_t7_24x40": (2, 1), "full_t8_64x64": (32, 2), "full_apm_t25_24x40": (8, 1)}


def check_grammar(wrapper, cfg):
    ref_u = {k: tuple(v.shape) for k, v in wrapper.diffusion_model.state_dict().items()}
    ref_c = {k: tuple(v.shape) for k, v in wrapper.controlnet.state_dict().items()}
    mine_u = arch.unet_param_shapes(cfg)
    mine_c = arch.controlnet_param_shapes(cfg)
    for name, ref, mine in (("unet", ref_u, mine_u), ("controlnet", ref_c, mine_c)):
        missing = sorted(set(ref) - set(mine))
        extra = sorted(set(mine) - set(ref))
        wrong = sorted(k for k in set(ref) & set(mine) if ref[k] != mine[k])
        assert not missing and not extra and not wrong, (
            f"{name} grammar mismatch: missing={missing[:5]} extra={extra[:5]} "
            f"wrong={[(k, ref[k], mine[k]) for k in wrong[:5]]}")
        print(f"  grammar {name}: {len(ref)} tensors, {sum(int(np.prod(s)) for s in ref.values()) / 1e6:.1f} M params OK")


def run_case(name, cfg, T, h, w, ctx_tokens, seed):
    print(f"[{name}] building reference modules ...", flush=True)
    torch.manual_seed(0)
    wrapper = ref_shims.build_reference(cfg)
    check_grammar(wrapper, cfg)
    sd_u = arch.synth_state_dict(arch.unet_param_shapes(cfg), seed=seed)
    sd_c = arch.synth_state_dict(arch.controlnet_param_shapes(cfg), seed=seed + 1000)
    wrapper.diffusion_model.load_state_dict(sd_u, strict=True)
    wrapper.controlnet.load_state_dict(sd_c, strict=True)
    x, t, c, kw = synth.make_inputs(cfg, T=T, h=h, w=w, seed=seed, ctx_tokens=ctx_tokens)

    captured = {}

    def hook(_m, _i, out):
        captured["hs"], captured["mid"] = out

    hd = wrapper.controlnet.register_forward_hook(hook)
    t0 = time.time()
    with torch.no_grad():
        ref_out = wrapper(x.clone(), t.clone(), {k: v.clone() for k, v in c.items()},
                          **{k: (v.clone() if torch.is_tensor(v) else v) for k, v in kw.items()})
    hd.remove()
    print(f"  reference forward {time.time() - t0:.1f}s  out absmax {ref_out.abs().max():.3f} std {ref_out.std():.3f}")

    taps = {}
    with torch.no_grad():
        my_out = orc.streaming_wrapper_forward(sd_u, sd_c, cfg, x, t, c, taps=taps, **kw)
    err = (my_out - ref_out).abs().max().item()
    err_mid = (taps["ctrl.middle"] - captured["mid"]).abs().max().item()
    err_hs = max((taps[f"ctrl.input_blocks.{i}"] - captured["hs"][i]).abs().max().item()
                 for i in range(len(captured["hs"])))
    print(f"  oracle vs reference: out {err:.3e}  ctrl.mid {err_mid:.3e}  ctrl.hs {err_hs:.3e}")
    scale = ref_out.abs().max().item()
    assert err <= 2e-4 * max(scale, 1.0), f"oracle restatement deviates from the reference: {err}"
    os.makedirs(GOLDEN, exist_ok=True)
    cstep, rstep = SAMPLING.get(name, (1, 1))
    np.savez_compressed(
        os.path.join(GOLDEN, f"streaming_{name}.npz"),
        out=ref_out[:, :, ::rstep].numpy().astype(np.float32),
        out_rstep=np.array([rstep], np.int64),
        ctrl_mid=captured["mid"][:, ::cstep].numpy().astype(np.float32),
        ctrl_hs_last=captured["hs"][-1][:, ::cstep].numpy().astype(np.float32),
        ctrl_cstep=np.array([cstep], np.int64),
        ctrl_hs0_stats=np.array([captured["hs"][0].mean().item(), captured["hs"][0].std().item()], np.float32),
        meta=np.array([T, h, w, ctx_tokens, seed, int(cfg.use_apm), cfg.model_channels], np.int64),
        oracle_vs_reference_maxerr=np.array([err, err_mid, err_hs], np.float64),
    )
    return err


if __name__ == "__main__":
    only = sys.argv[1:] or list(CASES)
    torch.set_num_threads(os.cpu_count() or 8)
    for name in only:
        run_case(name, *CASES[name])
    print("golden fixtures written to", GOLDEN)
