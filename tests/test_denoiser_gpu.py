"""End-to-end GPU parity of the denoiser seam (B200StreamingWrapper.forward == StreamingWrapper.forward).

Checked against (1) the committed golden vectors produced by the UNMODIFIED reference modules (tests/golden,
oracle/make_golden.py) and (2) the CPU oracle on the same seeded inputs, tap by tap.
Tolerance (bf16 activations + fp32 accumulate, vs the reference's fp32 CPU result): relative L2 <= 3e-2 on the
output latent update and on every block output; max-abs <= 6e-2 * max|ref|.  Measured on B200: see profiles/.
"""
import dataclasses
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
REL_TOL = 3e-2


def _rel(a, b):
    return ((a - b).norm() / b.norm()).item()


CASES = [("tiny_t8_16x16", False), ("tiny_t25_8x16", False), ("tiny_apm_t8_16x16", True), ("tiny_t7_24x40", False),
         # FULL network width (channel_mult (1,2,4,4)): BASELINE.json configs[0] (8 frames, 64x64 latent) and a
         # 25-frame APM case with odd extents; goldens from the unmodified reference (oracle/make_golden.py)
         ("full_t8_64x64", False), ("full_apm_t25_24x40", True)]


@pytest.mark.parametrize("name,apm", CASES)
def test_streaming_wrapper_vs_reference_golden(cuda_dev, name, apm):
    from oracle import streaming_svd_oracle as orc
    from streamingt2v_b200 import arch, synth
    from streamingt2v_b200.wrapper import B200StreamingWrapper
    g = np.load(os.path.join(GOLDEN, f"streaming_{name}.npz"))
    T, h, w, ctx_tokens, seed, use_apm, _ = (int(v) for v in g["meta"])
    base = arch.UNetConfig() if name.startswith("full") else arch.TINY
    cfg = dataclasses.replace(base, use_apm=bool(use_apm))
    cstep = int(g["ctrl_cstep"][0]) if "ctrl_cstep" in g else 1
    rstep = int(g["out_rstep"][0]) if "out_rstep" in g else 1         # latent rows kept of the output
    sd_u = arch.synth_state_dict(arch.unet_param_shapes(cfg), seed=seed)
    sd_c = arch.synth_state_dict(arch.controlnet_param_shapes(cfg), seed=seed + 1000)
    x, t, c, kw = synth.make_inputs(cfg, T=T, h=h, w=w, seed=seed, ctx_tokens=ctx_tokens)
    m = B200StreamingWrapper(cfg, sd_u, sd_c, cuda_dev)
    m.engine.debug_taps = {}
    xd, td = x.to(cuda_dev), t.to(cuda_dev)
    cd = {k: v.to(cuda_dev) for k, v in c.items()}
    kwd = {k: (v.to(cuda_dev) if torch.is_tensor(v) else v) for k, v in kw.items()}
    out = m(xd, td, cd, **kwd)
    torch.cuda.synchronize()
    out = out.float().cpu()
    assert torch.isfinite(out).all()
    ref = torch.from_numpy(g["out"])
    assert out[:, :, ::rstep].shape == ref.shape
    r = _rel(out[:, :, ::rstep], ref)
    mx = (out[:, :, ::rstep] - ref).abs().max().item()
    print(f"[{name}] out vs REFERENCE golden: rel_l2={r:.4e} max_abs={mx:.4e} ref_absmax={ref.abs().max():.3f}")
    # second call (exercises the cached conditioning path) must reproduce the first bit for bit
    out2 = m(xd, td, cd, **kwd).float().cpu()
    assert torch.equal(out, out2), "non-deterministic / stale cached conditioning"
    # tap-by-tap against the oracle
    taps = {}
    with torch.no_grad():
        o_ref = orc.streaming_wrapper_forward(sd_u, sd_c, cfg, x, t, c, taps=taps, **kw)
    assert _rel(o_ref[:, :, ::rstep], ref) < 1e-4  # the oracle itself reproduces the reference's golden output
    # so the whole output is held to the oracle with the golden's tolerance, rows the fixture does not store included
    assert _rel(out, o_ref) < REL_TOL and (out - o_ref).abs().max().item() < 6e-2 * o_ref.abs().max().item()
    worst = 0.0
    for tname, (tt, n, hh, ww) in m.engine.debug_taps.items():
        if tname in taps:
            mine = tt.float().cpu().reshape(n, hh, ww, -1).permute(0, 3, 1, 2)
            rr = _rel(mine, taps[tname])
            worst = max(worst, rr)
            print(f"   {tname:26s} rel_l2={rr:.4e}")
            assert rr < REL_TOL, f"{tname}: rel_l2 {rr}"
    mid = m.engine.debug_taps["ctrl.middle"]
    mid_t = mid[0].float().cpu().reshape(mid[1], mid[2], mid[3], -1).permute(0, 3, 1, 2)
    assert _rel(mid_t[:, ::cstep], torch.from_numpy(g["ctrl_mid"])) < REL_TOL
    assert r < REL_TOL and mx < 6e-2 * ref.abs().max().item()


def test_no_controlnet_path(cuda_dev):
    """hs_control_input=None branch of VideoUNet.forward (video_model.py:582-605): plain SVD denoiser (first chunk)."""
    from oracle import streaming_svd_oracle as orc
    from streamingt2v_b200 import arch, synth
    from streamingt2v_b200.model import B200Denoiser
    cfg = arch.TINY
    sd_u = arch.synth_state_dict(arch.unet_param_shapes(cfg), seed=7)
    x, t, c, kw = synth.make_inputs(cfg, T=8, h=8, w=8, seed=7)
    eng = B200Denoiser(cfg, sd_u, None, cuda_dev)
    out = eng.forward(x.to(cuda_dev), t.to(cuda_dev), {k: v.to(cuda_dev) for k, v in c.items()}, batch_size=2,
                      num_video_frames=8).float().cpu()
    with torch.no_grad():
        ref = orc.unet_forward(sd_u, cfg, torch.cat([x, c["concat"]], 1), t, c["crossattn"], c["vector"], 8, 7)
    r = _rel(out, ref)
    print(f"no-controlnet: rel_l2={r:.4e}")
    assert r < REL_TOL


def test_full_size_properties(cuda_dev):
    """BASELINE.json's full configuration (25 frames, 72x128 latent, CFG batch 2, full-width network), where the
    oracle is too slow to be the checker: size-independent properties of the seam instead.
      * finite and bit-for-bit deterministic;
      * the two videos of the batch never interact (every op on the path is per frame, per (video, pixel) or per
        video): changing video 1's inputs leaves video 0's output bit-identical and changes video 1's."""
    from streamingt2v_b200 import arch, synth
    from streamingt2v_b200.model import B200Denoiser
    cfg = arch.UNetConfig()
    T, h, w = 25, 72, 128
    eng = B200Denoiser(cfg, arch.synth_state_dict_device(arch.unet_param_shapes(cfg), cuda_dev, 1),
                       arch.synth_state_dict_device(arch.controlnet_param_shapes(cfg), cuda_dev, 2), cuda_dev)
    x, t, c, kw = synth.make_inputs(cfg, T=T, h=h, w=w, seed=5)
    x, t = x.to(cuda_dev), t.to(cuda_dev)
    c = {k: v.to(cuda_dev) for k, v in c.items()}
    ctrl = kw["ctrl_frames"].to(cuda_dev)

    def run():
        o = eng.forward(x, t, c, batch_size=2, num_video_frames=T, ctrl_frames=ctrl)
        torch.cuda.synchronize()
        return o.float().clone()

    o1 = run()
    assert o1.shape == (2 * T, 4, h, w) and bool(torch.isfinite(o1).all())
    assert float(o1.std()) > 0.0
    assert torch.equal(o1, run()), "full-size forward is not deterministic"
    x[T:].mul_(-0.5)                      # video 1 only (in place: the conditioning cache keys on tensor versions)
    c["concat"][T:].add_(0.25)
    c["crossattn"][T:].mul_(1.5)
    c["vector"][T:].mul_(-1.0)
    o3 = run()
    assert torch.equal(o3[:T], o1[:T]), "video 0 changed when only video 1's inputs changed"
    assert not torch.equal(o3[T:], o1[T:])


def test_conditioning_cache_recycled_storage(cuda_dev):
    """Freed-and-reallocated conditioning tensors of equal shape (the CUDA caching allocator hands the same address
    back) must not hit the step-invariant conditioning cache (round-1 finding)."""
    from streamingt2v_b200 import arch, synth
    from streamingt2v_b200.model import B200Denoiser
    cfg = arch.TINY
    T, h, w = 8, 8, 8
    eng = B200Denoiser(cfg, arch.synth_state_dict_fast(arch.unet_param_shapes(cfg), 3),
                       arch.synth_state_dict_fast(arch.controlnet_param_shapes(cfg), 4), cuda_dev)
    x, t, c, kw = synth.make_inputs(cfg, T=T, h=h, w=w, seed=5)
    x, t = x.to(cuda_dev), t.to(cuda_dev)

    def fresh(scale):
        cc = {k: (v * scale).to(cuda_dev) for k, v in c.items()}
        return cc, (kw["ctrl_frames"] * scale).to(cuda_dev)

    cc, ctrl = fresh(1.0)
    ptrs = [v.data_ptr() for v in cc.values()] + [ctrl.data_ptr()]
    outs = [eng.forward(x, t, cc, batch_size=2, num_video_frames=T, ctrl_frames=ctrl).clone()]
    same_addr = 0
    for i in range(1, 4):
        del cc, ctrl
        cc, ctrl = fresh(1.0 - 0.2 * i)
        same_addr += sum(a == b for a, b in zip(ptrs, [v.data_ptr() for v in cc.values()] + [ctrl.data_ptr()]))
        outs.append(eng.forward(x, t, cc, batch_size=2, num_video_frames=T, ctrl_frames=ctrl).clone())
        assert not torch.equal(outs[-1], outs[-2]), "stale conditioning served for new tensors"
    print(f"recycled addresses seen: {same_addr} (the cache keeps the keyed tensors alive, so 0 is expected)")
    # and against an engine that never cached anything: the last answer is the right one
    eng2 = B200Denoiser(cfg, arch.synth_state_dict_fast(arch.unet_param_shapes(cfg), 3),
                        arch.synth_state_dict_fast(arch.controlnet_param_shapes(cfg), 4), cuda_dev)
    ref = eng2.forward(x, t, cc, batch_size=2, num_video_frames=T, ctrl_frames=ctrl)
    assert torch.equal(ref, outs[-1])


def test_cuda_graph_replay_matches_eager(cuda_dev):
    """The recorded CUDA graph of the forward replays bit-for-bit what the eager launches compute, across steps (new
    x, t) and across chunks (new conditioning -> new recording)."""
    from streamingt2v_b200 import arch, synth
    from streamingt2v_b200.model import B200Denoiser
    cfg = arch.TINY
    T, h, w = 8, 16, 8
    sd_u = arch.synth_state_dict_fast(arch.unet_param_shapes(cfg), 3)
    sd_c = arch.synth_state_dict_fast(arch.controlnet_param_shapes(cfg), 4)
    eng_g = B200Denoiser(cfg, sd_u, sd_c, cuda_dev)
    eng_e = B200Denoiser(cfg, sd_u, sd_c, cuda_dev)
    eng_e.use_cuda_graph = False
    assert eng_g.use_cuda_graph
    x, t, c, kw = synth.make_inputs(cfg, T=T, h=h, w=w, seed=5)
    for chunk in range(2):
        cc = {k: (v * (1.0 + 0.1 * chunk)).to(cuda_dev) for k, v in c.items()}
        ctrl = (kw["ctrl_frames"] * (1.0 - 0.3 * chunk)).to(cuda_dev)
        for stepi in range(4):
            xs = (x * (1.0 + 0.05 * stepi)).to(cuda_dev)
            ts = (t - 0.1 * stepi).to(cuda_dev)
            a = eng_g.forward(xs, ts, cc, batch_size=2, num_video_frames=T, ctrl_frames=ctrl)
            b = eng_e.forward(xs, ts, cc, batch_size=2, num_video_frames=T, ctrl_frames=ctrl)
            assert torch.equal(a, b), (chunk, stepi)
    key = (2, T, h, w, True)
    assert eng_g._graphs[key]["graph"] is not None and eng_g._graphs[key]["launches"] > 100


def test_full_size_parity_vs_fp32_oracle_on_gpu(cuda_dev):
    """BASELINE.json's FULL configuration (25 frames, 72x128 latent, CFG batch 2, full-width network, ControlNet +
    CAM): the bf16 kernel path against the fp32 oracle — the restatement pinned to the unmodified reference on CPU
    (tests/test_oracle.py) — evaluated here on the GPU in fp32 (TF32 off) because 182 TFLOP is hours on host cores.
    The oracle is only the checker.  Same tolerance as the golden cases: rel-L2 <= 3e-2, max-abs <= 6e-2 max|ref|."""
    from oracle import streaming_svd_oracle as orc
    from streamingt2v_b200 import arch, synth
    from streamingt2v_b200.model import B200Denoiser
    cfg = arch.UNetConfig()
    T, h, w = 25, 72, 128
    sd_u = arch.synth_state_dict_device(arch.unet_param_shapes(cfg), cuda_dev, 1)
    sd_c = arch.synth_state_dict_device(arch.controlnet_param_shapes(cfg), cuda_dev, 2)
    eng = B200Denoiser(cfg, sd_u, sd_c, cuda_dev)
    x, t, c, kw = synth.make_inputs(cfg, T=T, h=h, w=w, seed=5)
    x, t = x.to(cuda_dev), t.to(cuda_dev)
    c = {k: v.to(cuda_dev) for k, v in c.items()}
    ctrl = kw["ctrl_frames"].to(cuda_dev)
    eng.debug_taps = {}
    out = eng.forward(x, t, c, batch_size=2, num_video_frames=T, ctrl_frames=ctrl).float()
    mine = {k: v for k, v in eng.debug_taps.items()}
    eng.debug_taps = None
    tf32 = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    try:
        taps = {}
        with torch.no_grad():
            ref = orc.streaming_wrapper_forward(sd_u, sd_c, cfg, x, t, c, batch_size=2, num_video_frames=T,
                                                ctrl_frames=ctrl, taps=taps)
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf32
    r = _rel(out, ref)
    mx = (out - ref).abs().max().item()
    print(f"[full size 25f 72x128] out vs fp32 oracle (GPU): rel_l2={r:.4e} max_abs={mx:.4e} "
          f"ref_absmax={ref.abs().max():.3f}")
    worst = ("", 0.0)
    for name, (tt, n, hh, ww) in mine.items():
        if name in taps:
            m = tt.float().reshape(n, hh, ww, -1).permute(0, 3, 1, 2)
            rr = _rel(m, taps[name])
            if rr > worst[1]:
                worst = (name, rr)
            assert rr < REL_TOL, f"{name}: rel_l2 {rr}"
    print(f"   worst tap: {worst[0]} rel_l2={worst[1]:.4e} over {len(mine)} taps")
    assert r < REL_TOL and mx < 6e-2 * ref.abs().max().item()
