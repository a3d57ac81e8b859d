"""Executed in a SUBPROCESS by tests/test_reference_callers_cpu.py (the kernels are swapped for the fp32 stand-ins of
tests/cpu_ops_emulation.py process-wide).

    python tests/run_reference_callers.py server  [keep|reencode]
    python tests/run_reference_callers.py classic

``server``  : harness/server_loop.py — the stand-in bench/smoke/GPU tests use — driving the drop-in classes for 4
              blocks, checked (a) against tests/golden/reference_callers_small.npz, what the UNMODIFIED
              ``release_server.GenerationSession`` computed on the same drop-ins with the same seed, draws and weights
              (tests/golden/make_reference_callers_golden.py): the same sequence of transformer / VAE calls with the same
              timesteps, cache positions and cache indices, and the same latents and pixels up to the CPU's summation
              order; and (b) against tests/golden/server_loop_small.npz, the same loop executed by the reference
              modules alone.
``classic`` : harness/classic_loop.py in place of the UNMODIFIED ``CausalInferencePipeline.inference``, checked the same
              way against the stored output of the reference pipeline and against tests/golden/pipeline_small.npz.
Prints one JSON line; exit code 0 = all assertions held.
"""
import json
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from tests import cpu_ops_emulation as emu  # noqa: E402
from tests.golden_io import ReplayRandn as Replay, load_npz, rel_l2, weights  # noqa: E402

DIMS = dict(dim=256, ffn_dim=512, num_heads=2, num_layers=2, text_dim=128)
W, H, NB = 96, 64, 4
PX_SUB = (Ellipsis, slice(None, None, 8), slice(None, None, 8))     # stored pixel sample: every 8th row and column
LAT_SUB = (Ellipsis, slice(None, None, 2), slice(None, None, 2))    # stored classic latents: every 2nd row and column
# Output tolerances against the stored caller output.  The same process computes it bit-equal; another CPU sums in
# another order and the bf16 / fp16 roundings then differ (measured with MKL and oneDNN restricted to AVX2: server
# latents 1.9e-3, pixels up to 2.7e-3; classic latents 1.2e-7, video 6.4e-4).  The call schedule is compared exactly.
TOL_SERVER, TOL_CLASSIC_LAT, TOL_CLASSIC_PX = 5e-3, 1e-4, 5e-3


def use_standin_kernels():
    import realtime_video_b200.dit as dit
    import realtime_video_b200.vae as vae
    import realtime_video_b200.wan_wrapper as ww
    for mod in (dit, ww, vae):
        mod.ops = emu


class CallTrace:
    """Records every call the loop makes into the drop-in classes, one int row per call (unused slots -1):
    transformer   [0, frames, current_start, kv global_end_index, kv local_end_index, crossattn is_init,
                   first timestep, last timestep]
    VAE decoder   [1, latent frames, cache entries set]
    VAE encoder   [2, frames, stream]
    classic VAE   [3, latent frames, use_cache]"""

    WIDTH = 8

    def __init__(self):
        self.rows = []

    def _add(self, *vals):
        self.rows.append([int(v) for v in vals] + [-1] * (self.WIDTH - len(vals)))

    def __enter__(self):
        import realtime_video_b200.vae as vae
        import realtime_video_b200.wan_wrapper as ww
        tr = self
        self._saved = [(ww.WanDiffusionWrapper, "forward"), (vae.VAEDecoderWrapper, "forward"),
                       (vae.VAEEncoderWrapper, "forward"), (ww.WanVAEWrapper, "decode_to_pixel")]
        self._saved = [(cls, name, cls.__dict__[name]) for cls, name in self._saved]
        f_dit, f_dec, f_enc, f_wan = (fn for _, _, fn in self._saved)

        def dit(self, noisy_image_or_video, conditional_dict, timestep, kv_cache=None, crossattn_cache=None,
                current_start=None, **kw):
            c0 = kv_cache[0]
            t = timestep.reshape(-1)
            tr._add(0, noisy_image_or_video.shape[1], current_start or 0, c0["global_end_index"],
                    c0["local_end_index"], bool(crossattn_cache[0]["is_init"]) if crossattn_cache else -1,
                    round(float(t[0])), round(float(t[-1])))
            return f_dit(self, noisy_image_or_video, conditional_dict, timestep, kv_cache, crossattn_cache,
                         current_start, **kw)

        def dec(self, z, *feat_cache):
            tr._add(1, z.shape[1], sum(c is not None for c in feat_cache))
            return f_dec(self, z, *feat_cache)

        def enc(self, z, feat_cache, stream=False):
            tr._add(2, z.shape[2], stream)
            return f_enc(self, z, feat_cache, stream)

        def wan(self, latent, use_cache=False):
            tr._add(3, latent.shape[1], use_cache)
            return f_wan(self, latent, use_cache)
        ww.WanDiffusionWrapper.forward, vae.VAEDecoderWrapper.forward = dit, dec
        vae.VAEEncoderWrapper.forward, ww.WanVAEWrapper.decode_to_pixel = enc, wan
        return self

    def __exit__(self, *exc):
        for cls, name, fn in self._saved:
            setattr(cls, name, fn)
        return False

    def array(self):
        return torch.tensor(self.rows, dtype=torch.int64).reshape(-1, self.WIDTH)


def fresh_server_models(g):
    """The drop-in models ``load_all`` (release_server.py:250-313) produces, from synthetic weights instead of
    checkpoints: transformer bf16 with fused projections (:176-177), VAE decoder / encoder fp16."""
    from realtime_video_b200.factory import synthetic_vae_params
    from realtime_video_b200.vae import VAEDecoderWrapper, VAEEncoderWrapper
    from realtime_video_b200.wan_wrapper import WanDiffusionWrapper
    tr = WanDiffusionWrapper(model_name="synthetic", timestep_shift=5.0, is_causal=True, model_config=dict(DIMS))
    tr.model.load_state_dict(weights(g, torch.bfloat16), strict=False)
    tr = tr.to(dtype=torch.bfloat16).eval().requires_grad_(False)
    for blk in tr.model.blocks:
        blk.self_attn.fuse_projections()
    dec = VAEDecoderWrapper()
    dec.load_state_dict(synthetic_vae_params(seed=0), strict=False)
    dec = dec.to(dtype=torch.float16).eval().requires_grad_(False)
    enc = VAEEncoderWrapper()
    enc.load_state_dict(synthetic_vae_params(seed=0, encoder=True), strict=False)
    enc = enc.to(dtype=torch.float16).eval().requires_grad_(False)
    return tr, dec, enc


def redirect_reencode_resize():
    """release_server.py:574 re-encodes at a hard-coded 480x832; redirect that literal resize to the test geometry
    (at 832x480 the bicubic resize is the identity), the same "patched-constant" device as the 1560."""
    import torch.nn.functional as F
    real_interp = F.interpolate

    def redirected(x, *a, **k):
        if k.get("size") is not None and tuple(k["size"]) == (480, 832):
            k["size"] = (H, W)
        return real_interp(x, *a, **k)
    F.interpolate = redirected


def classic_args():
    import types
    return types.SimpleNamespace(denoising_step_list=[1000, 750, 500, 250], warp_denoising_step=True,
                                 num_frame_per_block=3, independent_first_frame=False, context_noise=0,
                                 model_kwargs={})


def build_classic(cls, g, gd):
    """``cls`` (the reference's CausalInferencePipeline or harness.PipelineState) over the drop-in wrappers: the
    fixture DiT in fp32, the synthetic VAE in fp16."""
    from realtime_video_b200.factory import synthetic_vae_params
    from realtime_video_b200.wan_wrapper import WanDiffusionWrapper, WanVAEWrapper
    ctx = g["ctx"].float()
    gen = WanDiffusionWrapper(model_name="synthetic", timestep_shift=5.0, is_causal=True, model_config=dict(DIMS))
    gen.model.load_state_dict(weights(gd, torch.float32), strict=False)
    gen = gen.float().eval()
    vae = WanVAEWrapper(load_pretrained=False)
    vae.model.load_state_dict(synthetic_vae_params(seed=0), strict=False)
    vae = vae.half().eval()
    pipe = cls(classic_args(), "cpu", generator=gen, text_encoder=lambda text_prompts: {"prompt_embeds": ctx}, vae=vae)
    pipe.frame_seq_length = 96
    return pipe


def run_classic_pipe(pipe, g, twice=False):
    """``pipe.inference`` on the golden noise with the golden draws (twice: the second call goes through the
    reference's index-reset branch, causal_inference.py:123-133, 1-element tensors)."""
    real = torch.randn_like
    outs = []
    for _ in range(2 if twice else 1):
        it = iter([g[f"draw{i}"] for i in range(6)])
        torch.randn_like = lambda t, **kw: next(it).to(device=t.device, dtype=t.dtype)
        try:
            with torch.no_grad():
                outs.append(pipe.inference(g["noise"].float(), ["x"], return_latents=True))
        finally:
            torch.randn_like = real
    return outs


def run_server(mode: str) -> dict:
    keep = mode == "keep"
    use_standin_kernels()
    import harness
    g = load_npz("dit_small.npz")
    gold = load_npz("server_loop_small.npz")
    calls = load_npz("reference_callers_small.npz")
    tag = "keep" if keep else "reenc"
    draws = [gold[f"{tag}/draw{i}"] for i in range(int(gold[f"{tag}/ndraws"]))]
    pe = gold["prompt_embeds"]
    if not keep:
        redirect_reencode_resize()

    tr, dec, enc = fresh_server_models(g)
    hm = harness.build_models(tr, vae_decoder=dec, device="cpu", vae_encoder=enc)
    hp = harness.GenerateParams(width=W, height=H, seed=11, kv_cache_num_frames=3, num_blocks=NB,
                                num_denoising_steps=4, keep_first_frame=keep)
    with Replay(draws), CallTrace() as trace:
        hs = harness.GenerationSession(hp, hm, prompt_embeds=pe, device="cpu")
        h_px = [hs.generate_block().clone() for _ in range(NB)]
    assert hs.generate_block() is None and hs.block_idx == NB
    fs = (H // 16) * (W // 16)
    p = hm.pipeline
    assert list(p.kv_cache1[0]["k"].shape) == [1, 6 * fs, 2, 128]
    assert [p.kv_cache1[0]["global_end_index"], p.kv_cache1[0]["local_end_index"]] == [6 * fs, 6 * fs]
    assert [px.shape[1] for px in h_px] == calls[f"{tag}/frames"].tolist() == [6, 12, 12, 12]

    # (a) the unmodified GenerationSession on the same drop-ins, same seed / draws / weights
    want = calls[f"{tag}/trace"]
    got = trace.array()
    assert torch.equal(got, want), f"call sequence differs from the real GenerationSession:\n{got}\n{want}"
    out = {"mode": mode, "blocks": NB, "calls": len(got)}
    r = rel_l2(hs.all_latents.float(), calls[f"{tag}/latents"].float())
    out["latents_rel_l2_vs_caller"] = r
    assert r < TOL_SERVER, f"latents vs the real GenerationSession: rel_l2={r:.3e}"
    for b in range(NB):
        r = rel_l2(h_px[b][PX_SUB], calls[f"{tag}/px{b}"])
        out[f"px{b}_rel_l2_vs_caller"] = r
        assert r < TOL_SERVER, f"block {b} pixels vs the real GenerationSession: rel_l2={r:.3e}"

    # (b) the reference modules alone (golden): bf16 model / fp16 VAE on both sides, different arithmetic order
    r_lat = rel_l2(hs.all_latents.float(), gold[f"{tag}/latents"].float())
    out["latents_rel_l2"] = r_lat
    assert r_lat < 1e-2, f"latents vs reference-executed golden: rel_l2={r_lat:.3e}"
    for b in range(NB):
        ref = gold[f"{tag}/px{b}_sub"].float()
        got = h_px[b][..., ::2, ::2]
        assert got.shape == ref.shape, (got.shape, ref.shape)
        mad = (got - ref).abs().mean().item()
        out[f"px{b}_mad"] = mad
        assert mad < 6e-3, f"block {b} pixels vs golden: mean|d|={mad:.3e}"
    return out


def run_classic() -> dict:
    use_standin_kernels()
    import harness
    g, gd = load_npz("pipeline_small.npz"), load_npz("dit_small.npz")
    calls = load_npz("reference_callers_small.npz")
    with CallTrace() as trace:
        (hv, hl), (hv2, hl2) = run_classic_pipe(build_classic(harness.PipelineState, g, gd), g, twice=True)
    assert torch.equal(hl, hl2) and torch.equal(hv, hv2)
    # (a) the unmodified CausalInferencePipeline.inference on the same drop-ins, called twice the same way
    got, want = trace.array(), calls["classic/trace"]
    assert torch.equal(got, want), f"call sequence differs from the real CausalInferencePipeline:\n{got}\n{want}"
    r_lat = rel_l2(hl[LAT_SUB], calls["classic/latents"])
    r_px = rel_l2(hv[PX_SUB], calls["classic/video"])
    assert r_lat < TOL_CLASSIC_LAT and r_px < TOL_CLASSIC_PX, (r_lat, r_px)
    # (b) the reference modules alone (golden)
    r = rel_l2(hl, g["latents"])
    mad = (hv[..., ::2, ::2] - g["video_sub"]).abs().mean().item()
    assert r < 1e-3 and mad < 5e-3, (r, mad)
    return {"mode": "classic", "calls": len(got), "latents_rel_l2_vs_caller": r_lat, "video_rel_l2_vs_caller": r_px,
            "latents_rel_l2": r, "video_mad": mad}


if __name__ == "__main__":
    torch.set_num_threads(8)
    what = sys.argv[1]
    res = run_server(sys.argv[2]) if what == "server" else run_classic()
    print(json.dumps(res))
