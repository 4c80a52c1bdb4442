"""easyanimate_b200.pipelines (the reference's three pipeline call signatures without diffusers, loop on the fused sampler)
against the REFERENCE's own pipeline classes, both over the same product modules with the kernels replaced by the torch
stand-ins of tests/cpu_ops.py: same inputs, same seeded noise -> the same frames.  What differs between the two runs is only the
host code under test here (prompt plumbing, latent shapes, noise draw, conditioning preparation, schedule indexing, the fused
CFG + Euler update instead of four tensor ops, the fused output tail).  The reference pipelines' frames are stored results
(tests/refgold.py); on another CPU configuration they are matched within 3e-2 relative, three times the spread that the CPU
instruction set and thread count alone cause in these bf16 runs (below 1e-2)."""
import pytest
import torch

from oracle import dit, ref_pipeline, vae
from tests import cpu_ops, refgold

bf16 = torch.bfloat16
CFG = dict(num_attention_heads=2, attention_head_dim=64, in_channels=16, out_channels=16, patch_size=2, num_layers=2,
           time_embed_dim=64, add_norm_text_encoder=True, text_embed_dim=128, text_embed_dim_t5=None,
           time_position_encoding_type="3d_rope")
BOC = (64, 64, 128, 128)
H, W, FRAMES, LF, STEPS = 64, 96, 5, 2, 3


@pytest.fixture
def on_cpu(monkeypatch):
    import easyanimate_b200.autoencoder_magvit as A
    from easyanimate_b200 import ops
    cpu_ops.install(monkeypatch)
    cpu_ops.install_vae(monkeypatch)
    monkeypatch.setattr(ops, "cfg_euler_step", cpu_ops.cfg_euler_step)
    monkeypatch.setattr(A, "_require_cuda", lambda t, what: None)

    def decode_scaled(self, latents, out=None, dtype=torch.float32, to_host=False):  # no pinned memory / stream on this box
        self._latent_in_scale = 1.0 / float(self.config.scaling_factor)
        try:
            video = self._decode(latents)
        finally:
            self._latent_in_scale = 1.0
        return cpu_ops.frames_out(video.contiguous(), torch.empty(video.shape, dtype=dtype))

    monkeypatch.setattr(A.AutoencoderKLMagvit, "decode_scaled", decode_scaled)
    return A


def _modules(A, in_channels=16, seeds=(71, 72), **flags):
    from easyanimate_b200.transformer3d import EasyAnimateTransformer3DModel
    cfg = dict(CFG, in_channels=in_channels, **flags)
    ocfg = {k: v for k, v in cfg.items() if k not in flags and k != "time_position_encoding_type"}
    ob = dit.init_weights_(dit.OracleTransformer3D(**ocfg), seeds[0]).to(bf16)
    t = EasyAnimateTransformer3DModel(**cfg).to(bf16)
    t.load_state_dict(ob.state_dict(), strict=True)
    ov = vae.init_weights_(vae.OracleAutoencoderKLMagvit(block_out_channels=list(BOC), with_encoder=True), seeds[1]).to(bf16)
    v = A.AutoencoderKLMagvit(latent_channels=16, cache_mag_vae=True, spatial_group_norm=True, mid_block_attention_type="spatial",
                              block_out_channels=list(BOC), scaling_factor=0.7125, mini_batch_encoder=4, mini_batch_decoder=1).to(bf16)
    v.load_state_dict(ov.state_dict(), strict=True)
    return t, v


def _embeds(g):
    return (torch.randn(1, 9, 128, generator=g) * 3).to(bf16), (torch.randn(1, 9, 128, generator=g) * 3).to(bf16)


def _mask_kw(pe, ne):
    ones = torch.ones(pe.shape[:2], dtype=torch.long)
    return dict(prompt_embeds=pe, negative_prompt_embeds=ne, prompt_attention_mask=ones, negative_prompt_attention_mask=ones.clone(),
                prompt_embeds_2=pe, prompt_attention_mask_2=ones.clone())


def _same(got, want):
    assert got.dtype == torch.float32
    refgold.assert_equal(got, want, rel=3e-2)


def test_t2v_pipeline_equals_the_reference_pipeline(on_cpu):
    from easyanimate_b200 import EasyAnimatePipeline
    t, v = _modules(on_cpu)
    g = torch.Generator().manual_seed(1)
    lat = torch.randn(1, 16, LF, H // 8, W // 8, generator=g).to(bf16)
    pe, ne = _embeds(g)
    want = refgold.want("native/t2v", lambda: ref_pipeline.run(ref_pipeline.reference_pipeline(t, v), lat, pe, ne, height=H, width=W,
                                                               video_length=FRAMES, num_inference_steps=STEPS))
    pipe = EasyAnimatePipeline(vae=v, transformer=t)
    out = pipe(video_length=FRAMES, height=H, width=W, num_inference_steps=STEPS, guidance_scale=6.0, latents=lat, **_mask_kw(pe, ne))
    _same(out.frames, want)
    assert pipe.num_timesteps == STEPS and out[0] is out.frames
    # noise drawn by the pipeline itself: the reference's randn_tensor semantics (CPU generator, transformer dtype)
    want = refgold.want("native/t2v_generator", lambda: ref_pipeline.reference_pipeline(t, v)(
        video_length=FRAMES, height=H, width=W, num_inference_steps=2, guidance_scale=6.0, generator=torch.Generator().manual_seed(5),
        **_mask_kw(pe, ne)).frames)
    got = pipe(video_length=FRAMES, height=H, width=W, num_inference_steps=2, guidance_scale=6.0,
               generator=torch.Generator().manual_seed(5), **_mask_kw(pe, ne), output_type="numpy", return_dict=False)
    assert isinstance(got, __import__("numpy").ndarray)
    _same(torch.from_numpy(got), want)
    # no guidance (guidance_scale <= 1): one forward per step, no negative prompt needed
    want = refgold.want("native/t2v_no_guidance", lambda: ref_pipeline.reference_pipeline(t, v)(
        video_length=FRAMES, height=H, width=W, num_inference_steps=2, guidance_scale=1.0, latents=lat, **_mask_kw(pe, ne)).frames)
    _same(pipe(video_length=FRAMES, height=H, width=W, num_inference_steps=2, guidance_scale=1.0, latents=lat, **_mask_kw(pe, ne)).frames, want)


def test_t2v_pipeline_rejects_what_the_reference_rejects(on_cpu):
    from easyanimate_b200 import EasyAnimatePipeline
    t, v = _modules(on_cpu)
    pipe = EasyAnimatePipeline(vae=v, transformer=t)
    g = torch.Generator().manual_seed(2)
    pe, ne = _embeds(g)
    ok = dict(video_length=FRAMES, height=H, width=W, num_inference_steps=2, guidance_scale=6.0)
    bad_calls = [
        dict(ok, prompt_embeds=pe, prompt_attention_mask=torch.ones(1, 9)),                    # no prompt_embeds_2 (reference quirk)
        dict(ok, **{**_mask_kw(pe, ne), "prompt_attention_mask": None}),                       # embeds without their mask
        dict(ok, **{**_mask_kw(pe, ne), "negative_prompt_embeds": ne[:, :5]}),                 # shape mismatch
        dict(ok, prompt="a cat", **_mask_kw(pe, ne)),                                          # both prompt and embeds
        dict(ok, **_mask_kw(pe, ne), callback_on_step_end_tensor_inputs=["nope"]),
    ]
    def reference_errors():
        ref, errors = ref_pipeline.reference_pipeline(t, v), []
        for kw in bad_calls:
            with pytest.raises(ValueError) as e_ref:
                ref(**kw)
            errors.append(str(e_ref.value).split(":")[0][:40])
        return errors

    want = refgold.want("native/t2v_rejects", reference_errors)
    assert len(want) == len(bad_calls)
    for kw, e_ref in zip(bad_calls, want):
        with pytest.raises(ValueError) as e_ours:
            pipe(**kw)
        assert str(e_ours.value).split(":")[0][:40] == e_ref
    with pytest.raises(NotImplementedError):
        pipe(**ok, **_mask_kw(pe, ne), guidance_rescale=0.7)


def test_callback_on_step_end_sees_and_replaces_latents(on_cpu):
    from easyanimate_b200 import EasyAnimatePipeline
    t, v = _modules(on_cpu)
    g = torch.Generator().manual_seed(3)
    lat = torch.randn(1, 16, LF, H // 8, W // 8, generator=g).to(bf16)
    pe, ne = _embeds(g)
    seen = []

    def cb(pipe, i, t_, kw):
        seen.append((i, float(t_), tuple(kw["latents"].shape)))
        return {"latents": kw["latents"] * 0.5} if i == 0 else {}

    kw = dict(video_length=FRAMES, height=H, width=W, num_inference_steps=STEPS, guidance_scale=6.0, latents=lat, **_mask_kw(pe, ne))
    def reference_call():
        frames = ref_pipeline.reference_pipeline(t, v)(callback_on_step_end=cb, **kw).frames
        return {"frames": frames, "seen": list(seen)}

    want = refgold.want("native/callback", reference_call)
    seen[:] = []
    got = EasyAnimatePipeline(vae=v, transformer=t)(callback_on_step_end=cb, **kw).frames
    assert [[i, t_, list(s)] for i, t_, s in seen] == want["seen"] and len(seen) == STEPS
    want = want["frames"]
    _same(got, want)


@pytest.mark.parametrize("strength", [1.0, 0.7])
def test_inpaint_pipeline_equals_the_reference_pipeline(on_cpu, strength):
    from easyanimate_b200 import EasyAnimateInpaintPipeline
    t, v = _modules(on_cpu, in_channels=33, seeds=(73, 74), resize_inpaint_mask_directly=True, enable_clip_in_inpaint=False,
                    add_noise_in_inpaint_model=True)
    g = torch.Generator().manual_seed(4)
    video = torch.tile(torch.rand(1, 3, 1, H, W, generator=g), [1, 1, FRAMES, 1, 1])
    mask = torch.zeros_like(video[:, :1])
    mask[:, :, 1:] = 255
    pe, ne = _embeds(g)
    kw = dict(video_length=FRAMES, video=video, mask_video=mask, height=H, width=W, num_inference_steps=4, guidance_scale=6.0,
              strength=strength, noise_aug_strength=0.0563, **_mask_kw(pe, ne))
    want = refgold.want(f"native/inpaint_{strength}", lambda: ref_pipeline.reference_inpaint_pipeline(t, v)(
        generator=torch.Generator().manual_seed(9), **kw).frames)
    got = EasyAnimateInpaintPipeline(vae=v, transformer=t)(generator=torch.Generator().manual_seed(9), **kw).frames
    _same(got, want)


def test_inpaint_pipeline_all_masked_is_zero_conditioning(on_cpu):
    """mask == 255 everywhere: predict_t2v through the InP checkpoint (pipeline_easyanimate_inpaint.py:1322-1336)."""
    from easyanimate_b200 import EasyAnimateInpaintPipeline
    t, v = _modules(on_cpu, in_channels=33, seeds=(73, 74), resize_inpaint_mask_directly=True, enable_clip_in_inpaint=False)
    g = torch.Generator().manual_seed(6)
    video = torch.zeros(1, 3, FRAMES, H, W)
    mask = torch.full((1, 1, FRAMES, H, W), 255.0)
    pe, ne = _embeds(g)
    kw = dict(video_length=FRAMES, video=video, mask_video=mask, height=H, width=W, num_inference_steps=2, guidance_scale=6.0,
              **_mask_kw(pe, ne))
    want = refgold.want("native/inpaint_all_masked", lambda: ref_pipeline.reference_inpaint_pipeline(t, v)(
        generator=torch.Generator().manual_seed(10), **kw).frames)
    _same(EasyAnimateInpaintPipeline(vae=v, transformer=t)(generator=torch.Generator().manual_seed(10), **kw).frames, want)


@pytest.mark.parametrize("mode", ["control_video+ref", "control_video", "camera", "none"])
def test_control_pipeline_equals_the_reference_pipeline(on_cpu, mode):
    from easyanimate_b200 import EasyAnimateControlPipeline
    t, v = _modules(on_cpu, in_channels=48, seeds=(75, 76), add_ref_latent_in_control_model=True)
    g = torch.Generator().manual_seed(8)
    lat = torch.randn(1, 16, LF, H // 8, W // 8, generator=g).to(bf16)
    pe, ne = _embeds(g)
    kw = dict(video_length=FRAMES, height=H, width=W, num_inference_steps=STEPS, guidance_scale=6.0, latents=lat, **_mask_kw(pe, ne))
    if mode.startswith("control_video"):
        kw["control_video"] = torch.rand(1, 3, FRAMES, H, W, generator=g)
    if mode.endswith("+ref"):
        kw["ref_image"] = torch.rand(1, 3, 1, H, W, generator=g)
    if mode == "camera":
        kw["control_camera_video"] = torch.randn(1, 16, FRAMES, H, W, generator=g)
    want = refgold.want(f"native/control_{mode}", lambda: ref_pipeline.reference_control_pipeline(t, v)(**kw).frames)
    _same(EasyAnimateControlPipeline(vae=v, transformer=t)(**kw).frames, want)


class _FakeTokens(dict):
    input_ids = property(lambda self: self["input_ids"])
    attention_mask = property(lambda self: self["attention_mask"])

    def to(self, device):
        return self


class _FakeTokenizer:
    """Just enough of Qwen2Tokenizer for encode_prompt's LLM branch: a chat template and fixed-length 'tokens' (byte values)."""
    model_max_length = 32

    def apply_chat_template(self, messages, tokenize=False, add_generation_prompt=True):
        assert not tokenize and add_generation_prompt
        return "".join(f"<|user|>{m['content'][0]['text']}" for m in messages) + "<|assistant|>"

    def __call__(self, text, padding, max_length, truncation, return_attention_mask, padding_side, return_tensors):
        assert padding == "max_length" and truncation and return_attention_mask and padding_side == "right" and return_tensors == "pt"
        ids, mask = [], []
        for s in text:
            b = list(s.encode())[:max_length]
            ids.append(b + [0] * (max_length - len(b)))
            mask.append([1] * len(b) + [0] * (max_length - len(b)))
        return _FakeTokens(input_ids=torch.tensor(ids), attention_mask=torch.tensor(mask))


class _FakeTextEncoder(torch.nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.emb = torch.nn.Embedding(256, dim)
        self.mix = torch.nn.Linear(dim, dim)

    dtype = property(lambda self: self.emb.weight.dtype)
    device = property(lambda self: self.emb.weight.device)

    def forward(self, input_ids, attention_mask, output_hidden_states):
        assert output_hidden_states
        h0 = self.emb(input_ids) * attention_mask[..., None].to(self.dtype)
        h1 = self.mix(h0)
        return type("Out", (), {"hidden_states": [h0, h1, self.mix(h1)]})()


def test_prompt_strings_go_through_the_llm_branch_like_the_reference(on_cpu):
    """prompt / negative_prompt as strings: chat template -> tokenizer -> text_encoder(...).hidden_states[-2] -> the loop."""
    from easyanimate_b200 import EasyAnimatePipeline
    t, v = _modules(on_cpu)
    torch.manual_seed(0)
    tok, enc = _FakeTokenizer(), _FakeTextEncoder(128).to(bf16)
    lat = torch.randn(1, 16, LF, H // 8, W // 8, generator=torch.Generator().manual_seed(11)).to(bf16)
    kw = dict(prompt="a corgi surfing", negative_prompt="blurry", video_length=FRAMES, height=H, width=W, num_inference_steps=2,
              guidance_scale=6.0, latents=lat)

    def reference_call():
        ref = ref_pipeline.reference_pipeline(t, v)
        ref.tokenizer, ref.text_encoder = tok, enc
        frames = ref(**kw).frames
        return {"frames": frames, "embeds": ref.encode_prompt("a corgi surfing", torch.device("cpu"), bf16, negative_prompt="blurry")}

    want = refgold.want("native/prompt_strings", reference_call)
    got = EasyAnimatePipeline(vae=v, transformer=t, tokenizer=tok, text_encoder=enc)(**kw).frames
    _same(got, want["frames"])
    e_ours = EasyAnimatePipeline(vae=v, transformer=t, tokenizer=tok, text_encoder=enc).encode_prompt(
        "a corgi surfing", torch.device("cpu"), bf16, negative_prompt="blurry")
    assert len(e_ours) == len(want["embeds"])
    for a, b in zip(e_ours, want["embeds"]):
        refgold.assert_equal(a, b, rel=3e-2)


def test_teacache_inside_the_pipeline_call_matches_the_reference_pipeline(on_cpu):
    """predict_t2v.py:275-278 enables TeaCache on the transformer before calling the pipeline: the skip decisions are taken
    inside `transformer.forward`, so both pipelines see the same cached / computed steps and the same frames."""
    from easyanimate_b200 import EasyAnimatePipeline
    t, v = _modules(on_cpu)
    coeffs = [1.07862322, -4.19362456, 3.06725828, 0.33161686, 0.02374758]
    g = torch.Generator().manual_seed(21)
    lat = torch.randn(1, 16, LF, H // 8, W // 8, generator=g).to(bf16)
    pe, ne = _embeds(g)
    steps = 8
    kw = dict(video_length=FRAMES, height=H, width=W, num_inference_steps=steps, guidance_scale=6.0, latents=lat, **_mask_kw(pe, ne))
    t.enable_teacache(steps, 0.3, coefficients=coeffs)
    def reference_call():
        frames = ref_pipeline.reference_pipeline(t, v)(**kw).frames
        assert t.teacache.cnt == 0  # wrapped around after `steps` calls: ready for the next video
        return {"frames": frames, "skipped": t.teacache.skipped}

    want = refgold.want("native/teacache", reference_call)
    skipped_ref, want = want["skipped"], want["frames"]
    skipped0 = t.teacache.skipped
    got = EasyAnimatePipeline(vae=v, transformer=t)(**kw).frames
    assert 0 < skipped_ref < steps and t.teacache.skipped - skipped0 == skipped_ref and t.teacache.cnt == 0
    _same(got, want)


def test_two_videos_per_prompt(on_cpu):
    """num_images_per_prompt = 2: embeddings repeated, a batch of two latents (drawn at once, or from one generator per sample)."""
    from easyanimate_b200 import EasyAnimatePipeline
    t, v = _modules(on_cpu)
    pe, ne = _embeds(torch.Generator().manual_seed(31))
    kw = dict(video_length=FRAMES, height=H, width=W, num_inference_steps=2, guidance_scale=6.0, num_images_per_prompt=2,
              **_mask_kw(pe, ne))
    pipe = EasyAnimatePipeline(vae=v, transformer=t)
    want = refgold.want("native/two_videos", lambda: ref_pipeline.reference_pipeline(t, v)(
        generator=torch.Generator().manual_seed(32), **kw).frames)
    got = pipe(generator=torch.Generator().manual_seed(32), **kw).frames
    assert got.shape == (2, 3, FRAMES, H, W)
    _same(got, want)
    with pytest.raises(ValueError, match="list of generators"):
        pipe(generator=[torch.Generator().manual_seed(1)] * 3, **kw)


def test_load_pipeline_follows_the_predict_scripts_loading_sequence(on_cpu, tmp_path):
    """predict_t2v.py:94-255 on a released-layout directory (transformer/, vae/, scheduler/ with config.json + safetensors):
    `load_pipeline` returns the pipeline class the scripts pick (InP checkpoint -> inpaint pipeline), with the scheduler of
    scheduler_config.json, and its call equals the call of a pipeline built by hand from the same weights."""
    import json
    from safetensors.torch import save_file
    from easyanimate_b200 import EasyAnimateInpaintPipeline, EasyAnimatePipeline, load_pipeline
    t, v = _modules(on_cpu, in_channels=33, seeds=(91, 92), resize_inpaint_mask_directly=True, enable_clip_in_inpaint=False)
    for name, module in (("transformer", t), ("vae", v)):
        d = tmp_path / name
        d.mkdir()
        (d / "config.json").write_text(json.dumps(dict(module.config)))
        save_file({k: x.detach().contiguous() for k, x in module.state_dict().items()}, str(d / "diffusion_pytorch_model.safetensors"))
    (tmp_path / "scheduler").mkdir()
    (tmp_path / "scheduler" / "scheduler_config.json").write_text(json.dumps(
        {"_class_name": "FlowMatchEulerDiscreteScheduler", "_diffusers_version": "0.31.0", "num_train_timesteps": 1000, "shift": 3.0,
         "use_dynamic_shifting": False, "base_shift": 0.5, "max_shift": 1.15, "base_image_seq_len": 256, "max_image_seq_len": 4096}))
    pipe = load_pipeline(str(tmp_path), device="cpu")
    assert isinstance(pipe, EasyAnimateInpaintPipeline) and pipe.scheduler.config.shift == 3.0 and pipe.tokenizer is None
    assert pipe.transformer.dtype == bf16 and pipe.transformer.resize_inpaint_mask_directly and pipe.vae.cache_mag_vae
    for k, x in t.state_dict().items():
        assert torch.equal(pipe.transformer.state_dict()[k], x), k
    g = torch.Generator().manual_seed(93)
    video = torch.tile(torch.rand(1, 3, 1, H, W, generator=g), [1, 1, FRAMES, 1, 1])
    mask = torch.zeros_like(video[:, :1])
    mask[:, :, 1:] = 255
    pe, ne = _embeds(g)
    kw = dict(video_length=FRAMES, video=video, mask_video=mask, height=H, width=W, num_inference_steps=2, guidance_scale=6.0,
              **_mask_kw(pe, ne))
    from easyanimate_b200 import FlowMatchEulerDiscreteScheduler
    by_hand = EasyAnimateInpaintPipeline(vae=v, transformer=t, scheduler=FlowMatchEulerDiscreteScheduler(shift=3.0))
    a, b = pipe(generator=torch.Generator().manual_seed(94), **kw).frames, by_hand(generator=torch.Generator().manual_seed(94), **kw).frames
    assert a.dtype == b.dtype == torch.float32 and torch.equal(a, b), float((a - b).abs().max())
    # a 16-channel checkpoint gives the text-to-video pipeline
    t16, _ = _modules(on_cpu, seeds=(95, 92))
    (tmp_path / "transformer" / "config.json").write_text(json.dumps(dict(t16.config)))
    save_file({k: x.detach().contiguous() for k, x in t16.state_dict().items()},
              str(tmp_path / "transformer" / "diffusion_pytorch_model.safetensors"))
    assert type(load_pipeline(str(tmp_path), device="cpu")) is EasyAnimatePipeline


@pytest.mark.parametrize("video_length,h,w", [(1, 64, 96), (9, 48, 80), (5, 70, 100)])
def test_t2v_edge_shapes(on_cpu, video_length, h, w):
    """A single image (video_length 1 -> one latent frame), 1 + 8 frames, and a size that is not a multiple of 16 (both pipelines
    round it down: pipeline_easyanimate.py:874-876)."""
    from easyanimate_b200 import EasyAnimatePipeline
    t, v = _modules(on_cpu)
    pe, ne = _embeds(torch.Generator().manual_seed(41))
    kw = dict(video_length=video_length, height=h, width=w, num_inference_steps=2, guidance_scale=6.0, **_mask_kw(pe, ne))
    want = refgold.want(f"native/edge_{video_length}x{h}x{w}", lambda: ref_pipeline.reference_pipeline(t, v)(
        generator=torch.Generator().manual_seed(42), **kw).frames)
    got = EasyAnimatePipeline(vae=v, transformer=t)(generator=torch.Generator().manual_seed(42), **kw).frames
    assert got.shape == (1, 3, video_length, h // 16 * 16, w // 16 * 16)
    _same(got, want)


def test_inpaint_pipeline_with_vae_encoded_mask(on_cpu):
    """resize_inpaint_mask_directly = False (EasyAnimate V5 InP: 16 + 16 + 16 input channels): the mask itself goes through
    `vae.encode` (pipeline_easyanimate_inpaint.py:1364-1376, 781-792) instead of being resized."""
    from easyanimate_b200 import EasyAnimateInpaintPipeline
    t, v = _modules(on_cpu, in_channels=48, seeds=(77, 78), resize_inpaint_mask_directly=False, enable_clip_in_inpaint=False)
    g = torch.Generator().manual_seed(14)
    video = torch.rand(1, 3, FRAMES, H, W, generator=g)
    mask = torch.zeros_like(video[:, :1])
    mask[:, :, 2:, :, W // 2:] = 255
    pe, ne = _embeds(g)
    kw = dict(video_length=FRAMES, video=video, mask_video=mask, height=H, width=W, num_inference_steps=2, guidance_scale=6.0,
              **_mask_kw(pe, ne))
    want = refgold.want("native/inpaint_vae_mask", lambda: ref_pipeline.reference_inpaint_pipeline(t, v)(
        generator=torch.Generator().manual_seed(15), **kw).frames)
    _same(EasyAnimateInpaintPipeline(vae=v, transformer=t)(generator=torch.Generator().manual_seed(15), **kw).frames, want)


def test_inpaint_reference_video_noise_with_sampled_strength(on_cpu):
    """noise_aug_strength = None: one noise level per sample drawn from exp(N(-3, 0.5)) with the GLOBAL generator
    (pipeline_easyanimate_inpaint.py:153-157), then the noise itself with the call's generator."""
    from easyanimate_b200 import EasyAnimateInpaintPipeline
    t, v = _modules(on_cpu, in_channels=33, seeds=(73, 74), resize_inpaint_mask_directly=True, enable_clip_in_inpaint=False,
                    add_noise_in_inpaint_model=True)
    g = torch.Generator().manual_seed(16)
    video = torch.rand(1, 3, FRAMES, H, W, generator=g)
    mask = torch.zeros_like(video[:, :1])
    mask[:, :, 1:] = 255
    pe, ne = _embeds(g)
    kw = dict(video_length=FRAMES, video=video, mask_video=mask, height=H, width=W, num_inference_steps=2, guidance_scale=6.0,
              noise_aug_strength=None, **_mask_kw(pe, ne))
    torch.manual_seed(17)
    want = refgold.want("native/inpaint_sampled_strength", lambda: ref_pipeline.reference_inpaint_pipeline(t, v)(
        generator=torch.Generator().manual_seed(18), **kw).frames)
    torch.manual_seed(17)
    got = EasyAnimateInpaintPipeline(vae=v, transformer=t)(generator=torch.Generator().manual_seed(18), **kw).frames
    _same(got, want)
