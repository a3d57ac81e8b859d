"""Golden for tests/test_reference_callers_cpu.py: what the reference's OWN callers compute, unmodified, on the drop-in
classes (kernels replaced by the fp32 stand-ins of tests/cpu_ops_emulation.py).  Needs the reference checkout
(tests/ref_env.py); the test itself runs without it.

    python tests/golden/make_reference_callers_golden.py      # writes tests/golden/reference_callers_small.npz

* ``keep`` / ``reenc``: ``release_server.GenerationSession`` (``__init__`` -> ``init_models`` ->
  ``generate_block_internal`` x 4: recompute_kv_cache, get_clean_context_frames, denoise loop, VAE decode, sliding
  window) on the models ``load_all`` would build, 96x64, the draws of server_loop_small.npz;
* ``classic``: ``CausalInferencePipeline.inference`` called twice on the drop-in wrappers (pipeline_small.npz).

Stored per case: the call sequence into the drop-in classes (run_reference_callers.CallTrace), the latents (all of
them as bf16 bits for the server; every 2nd row and column, fp32, for the classic pipeline) and the pixels sampled at
every 8th row and column, fp32.  Each case also runs harness/ (the stand-in the GPU tests and bench.py drive) in the
same process and asserts it is bit-equal.
"""
import sys
import types
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
sys.path.insert(0, str(ROOT))
from tests import ref_env  # noqa: E402
from tests import run_reference_callers as rc  # noqa: E402
from tests.golden_io import ReplayRandn as Replay, load_npz, rel_l2  # noqa: E402

OUT = {}


def bf16_bits(t):
    return t.detach().contiguous().view(torch.int16).numpy()


def server(mode: str):
    keep = mode == "keep"
    tag = "keep" if keep else "reenc"
    rs = ref_env.setup(dropin=True)
    rc.use_standin_kernels()
    from demo_utils.vae_block3 import VAEDecoderWrapper
    from pipeline import CausalInferencePipeline          # the reference's own pipeline class
    from utils.wan_wrapper import WanDiffusionWrapper

    import realtime_video_b200.vae as vae
    import realtime_video_b200.wan_wrapper as ww
    assert WanDiffusionWrapper is ww.WanDiffusionWrapper and VAEDecoderWrapper is vae.VAEDecoderWrapper
    assert CausalInferencePipeline.__module__ == "pipeline.causal_inference" and \
        "reference" in sys.modules["pipeline.causal_inference"].__file__
    g = load_npz("dit_small.npz")
    gold = load_npz("server_loop_small.npz")
    draws = [gold[f"{tag}/draw{i}"] for i in range(int(gold[f"{tag}/ndraws"]))]
    pe = gold["prompt_embeds"]
    if not keep:
        rc.redirect_reencode_resize()

    class StaticText(torch.nn.Module):
        def forward(self, text_prompts):
            return {"prompt_embeds": pe.clone()}
    text = StaticText()
    tr, dec, enc = rc.fresh_server_models(g)
    pipe = CausalInferencePipeline(rc.classic_args(), device="cpu", generator=tr, text_encoder=text, vae=dec)
    pipe.frame_seq_length = (rc.H // 16) * (rc.W // 16)      # INTEGRATION.md: other resolutions than 832x480
    models = rs.Models(text, tr, pipe, enc, dec)

    frames_cb = []
    params = rs.GenerateParams(prompt="x", width=rc.W, height=rc.H, seed=11, kv_cache_num_frames=3,
                               num_blocks=rc.NB, num_denoising_steps=4, keep_first_frame=keep)
    with Replay(draws), rc.CallTrace() as trace:
        sess = rs.GenerationSession(params, types.SimpleNamespace(use_taehv=False),
                                    frame_callback=lambda px, ids, ev: frames_cb.append(px.shape[1]), models=models)
        assert type(sess).__module__ == "release_server"
        real_px = [sess.generate_block_internal(models).clone() for _ in range(rc.NB)]
    assert sess.generate_block_internal(models) is None and sess.block_idx == rc.NB
    assert frames_cb == [6, 12, 12, 12]

    # harness/ in the same process: bit-equal, call for call
    import harness
    tr2, dec2, enc2 = rc.fresh_server_models(g)
    hm = harness.build_models(tr2, vae_decoder=dec2, device="cpu", vae_encoder=enc2)
    hp = harness.GenerateParams(width=rc.W, height=rc.H, seed=11, kv_cache_num_frames=3, num_blocks=rc.NB,
                                num_denoising_steps=4, keep_first_frame=keep)
    with Replay(draws), rc.CallTrace() as htrace:
        hs = harness.GenerationSession(hp, hm, prompt_embeds=pe, device="cpu")
        h_px = [hs.generate_block().clone() for _ in range(rc.NB)]
    assert torch.equal(trace.array(), htrace.array())
    assert all(torch.equal(a, b) for a, b in zip(real_px, h_px)) and torch.equal(sess.all_latents, hs.all_latents)

    OUT[f"{tag}/trace"] = trace.array().numpy()
    OUT[f"{tag}/frames"] = np.array(frames_cb)
    OUT[f"{tag}/latents@bf16"] = bf16_bits(sess.all_latents)
    for b, px in enumerate(real_px):
        OUT[f"{tag}/px{b}"] = px[rc.PX_SUB].float().contiguous().numpy()
    print(tag, len(trace.rows), "calls; latents vs reference-only golden",
          rel_l2(sess.all_latents.float(), gold[f"{tag}/latents"].float()), flush=True)
    ref_env.teardown()
    torch.set_grad_enabled(True)


def classic():
    ref_env.setup(dropin=True)
    rc.use_standin_kernels()
    from pipeline import CausalInferencePipeline

    import harness
    g, gd = load_npz("pipeline_small.npz"), load_npz("dit_small.npz")
    ref_pipe = rc.build_classic(CausalInferencePipeline, g, gd)
    assert "reference" in sys.modules[type(ref_pipe).__module__].__file__
    with rc.CallTrace() as trace:
        (v1, l1), (v2, l2) = rc.run_classic_pipe(ref_pipe, g, twice=True)
    assert torch.equal(l1, l2) and torch.equal(v1, v2)
    with rc.CallTrace() as htrace:
        (hv, hl), _ = rc.run_classic_pipe(rc.build_classic(harness.PipelineState, g, gd), g, twice=True)
    assert torch.equal(trace.array(), htrace.array()) and torch.equal(l1, hl) and torch.equal(v1, hv)
    OUT["classic/trace"] = trace.array().numpy()
    OUT["classic/latents"] = l1[rc.LAT_SUB].float().contiguous().numpy()
    OUT["classic/video"] = v1[rc.PX_SUB].float().contiguous().numpy()
    print("classic", len(trace.rows), "calls; latents vs reference-only golden", rel_l2(l1, g["latents"]), flush=True)
    ref_env.teardown()


if __name__ == "__main__":
    torch.set_num_threads(8)
    server("keep")
    server("reencode")
    classic()
    np.savez_compressed(HERE / "reference_callers_small.npz", **OUT)
    print("reference_callers_small.npz", sum(v.nbytes for v in OUT.values()) / 1e6, "MB raw")
