"""SURVEY.md section 8b, the boundary's strongest proof available without a GPU: the REFERENCE's own pipeline classes
(easyanimate/pipeline/pipeline_easyanimate.py:769-1148 and its inpaint / control siblings, executed unmodified through
oracle/ref_pipeline.py where the original project is installed) over the reference's own transformer + VAE, whose frames are
stored (tests/refgold.py) and

  (1) pin oracle.dit.denoise_loop + oracle.vae decode + the decode_latents tail (what every GPU parity test compares with)
      against the reference's loop, not against a restatement of it;
  (2) are what the PRODUCT pipelines over the PRODUCT modules (easyanimate_b200.EasyAnimateTransformer3DModel /
      AutoencoderKLMagvit, kernels replaced by the torch stand-ins of tests/cpu_ops.py) produce from the same call, up to bf16
      round-off; tests/test_native_pipelines_cpu.py pins the product pipelines to the reference's over the same modules.

The GPU-side counterpart is the fixture `pipe_ref_t2v.safetensors` minted by (1) (tests/golden/make_golden.py) and compared with
in tests/test_pipeline_gpu.py."""
import pytest
import torch

from oracle import dit, ref_pipeline, vae
from tests import refgold
from tests.test_native_pipelines_cpu import on_cpu  # noqa: F401  (fixture: product modules on the torch stand-ins)

bf16 = torch.bfloat16
CFG = dict(num_attention_heads=2, attention_head_dim=64, in_channels=16, out_channels=16, patch_size=2, num_layers=2,
           time_embed_dim=64, add_norm_text_encoder=True, text_embed_dim=128, text_embed_dim_t5=None)
BOC = (64, 64, 128, 128)
H, W, FRAMES, LF, STEPS = 64, 96, 5, 2, 3


def _inputs(seed=5):
    g = torch.Generator().manual_seed(seed)
    lat = torch.randn(1, 16, LF, H // 8, W // 8, generator=g)
    pe, ne = torch.randn(1, 9, 128, generator=g) * 3, torch.randn(1, 9, 128, generator=g) * 3
    return lat, pe, ne


def _reference_modules(dtype):
    from oracle import ref_dit, ref_vae
    rt = ref_dit.reference_transformer(**CFG, time_position_encoding_type="3d_rope").eval()
    rt.load_state_dict(dit.init_weights_(dit.OracleTransformer3D(**CFG), 31).state_dict(), strict=True)
    rv = ref_vae.reference_autoencoder(block_out_channels=BOC).eval()
    rv.load_state_dict(vae.init_weights_(vae.OracleAutoencoderKLMagvit(block_out_channels=list(BOC)), 32).state_dict(), strict=False)
    return rt.to(dtype), rv.to(dtype)


def _oracle_frames(lat, pe, ne, dtype):
    ot = dit.init_weights_(dit.OracleTransformer3D(**CFG), 31).to(dtype)
    ov = vae.init_weights_(vae.OracleAutoencoderKLMagvit(block_out_channels=list(BOC)), 32).to(dtype)
    with torch.no_grad():
        z = dit.denoise_loop(ot, lat.to(dtype), pe.to(dtype), ne.to(dtype), dit.rope_for_video(H, W, LF), num_steps=STEPS,
                             guidance_scale=6.0)
        video = ov.decode(1 / ov.scaling_factor * z)[0].clamp(-1, 1)
        return z, (video / 2 + 0.5).clamp(0, 1).float()


def test_reference_pipeline_call_pins_the_oracle_loop_fp32():
    lat, pe, ne = _inputs()
    frames = refgold.want("ref_pipeline/fp32", lambda: ref_pipeline.run(
        ref_pipeline.reference_pipeline(*_reference_modules(torch.float32)), lat, pe, ne, height=H, width=W, video_length=FRAMES,
        num_inference_steps=STEPS))
    _, want = _oracle_frames(lat, pe, ne, torch.float32)
    assert frames.shape == want.shape == (1, 3, FRAMES, H, W) and frames.dtype == str(want.dtype)
    refgold.assert_close(want, frames, atol=2e-5)  # two fp32 evaluations of the same graph


def test_reference_pipeline_call_pins_the_oracle_loop_bf16():
    """In bf16 the loop's rounding points matter (timestep to bf16, CFG combine in bf16, (sigma_next - sigma) rounded to bf16
    by type promotion, fp32 sample): the oracle's loop reproduces the reference pipeline's latents bit for bit."""
    lat, pe, ne = _inputs(6)

    def reference_call():
        pipe = ref_pipeline.reference_pipeline(*_reference_modules(bf16))
        seen = {}
        orig = pipe.decode_latents
        pipe.decode_latents = lambda z: (seen.setdefault("z", z.clone()), orig(z))[1]
        frames = ref_pipeline.run(pipe, lat.to(bf16), pe.to(bf16), ne.to(bf16), height=H, width=W, video_length=FRAMES,
                                  num_inference_steps=STEPS)
        return {"z": seen["z"], "frames": frames}

    ref = refgold.want("ref_pipeline/bf16", reference_call)
    z, want = _oracle_frames(lat, pe, ne, bf16)
    refgold.assert_equal(z, ref["z"], rel=3e-2)
    refgold.assert_close(want, ref["frames"], atol=2e-2, elsewhere_rel=3e-2)


def test_reference_pipeline_drives_the_product_modules(on_cpu):
    from easyanimate_b200 import EasyAnimatePipeline
    from easyanimate_b200.transformer3d import EasyAnimateTransformer3DModel
    AutoencoderKLMagvit = on_cpu.AutoencoderKLMagvit
    lat, pe, ne = (t.to(bf16) for t in _inputs(7))
    ob = dit.init_weights_(dit.OracleTransformer3D(**CFG), 31).to(bf16)
    ours_t = EasyAnimateTransformer3DModel(**CFG, time_position_encoding_type="3d_rope").to(bf16)
    ours_t.load_state_dict(ob.state_dict(), strict=True)
    ov = vae.init_weights_(vae.OracleAutoencoderKLMagvit(block_out_channels=list(BOC)), 32).to(bf16)
    ours_v = AutoencoderKLMagvit(latent_channels=16, cache_mag_vae=True, spatial_group_norm=True,
                                 mid_block_attention_type="spatial", block_out_channels=list(BOC), scaling_factor=0.7125).to(bf16)
    ours_v.load_state_dict(ov.state_dict(), strict=False)
    frames = ref_pipeline.run(EasyAnimatePipeline(vae=ours_v, transformer=ours_t), lat, pe, ne, height=H, width=W,
                              video_length=FRAMES, num_inference_steps=STEPS)
    want = refgold.want("ref_pipeline/t2v_reference_modules", lambda: ref_pipeline.run(
        ref_pipeline.reference_pipeline(*_reference_modules(bf16)), lat, pe, ne, height=H, width=W, video_length=FRAMES,
        num_inference_steps=STEPS))
    assert tuple(frames.shape) == want.shape == (1, 3, FRAMES, H, W) and frames.dtype == torch.float32
    rel = refgold.diff(frames, want)[1]
    assert rel < 3e-2, rel  # bf16 round-off of two op orders through 3 CFG steps + decode; a plumbing error is O(1)


# ---- a17: the I2V path through the reference's own EasyAnimateInpaintPipeline (predict_i2v.py) -------------------------------
I2V_CFG = dict(CFG, in_channels=33, time_position_encoding_type="3d_rope", resize_inpaint_mask_directly=True,
               enable_clip_in_inpaint=False, add_noise_in_inpaint_model=True)


def _i2v_inputs(seed=9):
    g = torch.Generator().manual_seed(seed)
    first = torch.rand(1, 3, 1, H, W, generator=g)
    video = torch.tile(first, [1, 1, FRAMES, 1, 1])                 # utils.py:105-110: the start image on every frame, in [0, 1]
    mask = torch.zeros_like(video[:, :1])
    mask[:, :, 1:] = 255                                             # frame 0 is given, the rest is to be generated
    pe, ne = torch.randn(1, 9, 128, generator=g) * 3, torch.randn(1, 9, 128, generator=g) * 3
    return video, mask, pe, ne


def test_reference_inpaint_pipeline_drives_the_product_modules(on_cpu):
    """`EasyAnimateInpaintPipeline.__call__` (pipeline_easyanimate_inpaint.py:978-1604): VaeImageProcessor -> masked video ->
    `vae.encode(...)[0].mode()` * scaling_factor -> resize_mask -> inpaint_latents (1 + 16 channels) -> denoise loop with
    `inpaint_latents=` -> decode_latents.  The reference's class over the reference's transformer + VAE (stored), the product's
    over the product's (kernels = torch stand-ins): same start noise (seeded generator), same frames up to bf16 round-off."""
    from easyanimate_b200 import EasyAnimateInpaintPipeline
    from easyanimate_b200.transformer3d import EasyAnimateTransformer3DModel
    A = on_cpu
    video, mask, pe, ne = _i2v_inputs()
    pe, ne = pe.to(bf16), ne.to(bf16)
    ocfg = {k: v for k, v in I2V_CFG.items() if k in CFG}
    ob = dit.init_weights_(dit.OracleTransformer3D(**ocfg), 51).to(bf16)
    ov = vae.init_weights_(vae.OracleAutoencoderKLMagvit(block_out_channels=list(BOC), with_encoder=True), 52).to(bf16)

    def reference_call():
        from oracle import ref_dit, ref_vae
        rt = ref_dit.reference_transformer(**I2V_CFG).eval()
        rt.load_state_dict(ob.state_dict(), strict=True)
        rv = ref_vae.reference_autoencoder(block_out_channels=BOC).eval()
        rv.load_state_dict(ov.state_dict(), strict=True)
        return ref_pipeline.run_inpaint(ref_pipeline.reference_inpaint_pipeline(rt.to(bf16), rv.to(bf16)), video, mask, pe, ne,
                                        height=H, width=W, num_inference_steps=STEPS, seed=77)

    want = refgold.want("ref_pipeline/inpaint_reference_modules", reference_call)

    ours_t = EasyAnimateTransformer3DModel(**I2V_CFG).to(bf16)
    ours_t.load_state_dict(ob.state_dict(), strict=True)
    ours_v = A.AutoencoderKLMagvit(latent_channels=16, cache_mag_vae=True, spatial_group_norm=True, mid_block_attention_type="spatial",
                                   block_out_channels=list(BOC), scaling_factor=0.7125, mini_batch_encoder=4,
                                   mini_batch_decoder=1).to(bf16)
    ours_v.load_state_dict(ov.state_dict(), strict=True)
    seen = {}
    enc = ours_v.encode
    ours_v.encode = lambda x, *a, **k: (seen.setdefault("encode_calls", []).append(tuple(x.shape)), enc(x, *a, **k))[1]
    frames = ref_pipeline.run_inpaint(EasyAnimateInpaintPipeline(vae=ours_v, transformer=ours_t), video, mask, pe, ne,
                                      height=H, width=W, num_inference_steps=STEPS, seed=77)
    assert seen["encode_calls"] == [(1, 3, FRAMES, H, W)]  # the masked video, once (resize_inpaint_mask_directly: no mask encode)
    assert tuple(frames.shape) == want.shape == (1, 3, FRAMES, H, W) and frames.dtype == torch.float32
    rel = refgold.diff(frames, want)[1]
    assert rel < 3e-2, rel


# ---- f4: the Control path through the reference's own EasyAnimateControlPipeline ---------------------------------------------
CONTROL_CFG = dict(CFG, in_channels=48, time_position_encoding_type="3d_rope", add_ref_latent_in_control_model=True)


@pytest.mark.parametrize("with_ref_image", [True, False])
def test_reference_control_pipeline_drives_the_product_modules(on_cpu, with_ref_image):
    """`EasyAnimateControlPipeline.__call__` (pipeline_easyanimate_control.py:833-1282): control video -> `vae.encode` ->
    control_latents (16 channels) + the reference image's latent in frame 0 of 16 more channels (add_ref_latent_in_control_model)
    -> `transformer(..., control_latents=)` -> decode_latents.  The reference's class over the reference's modules (stored), the
    product's over the product's."""
    from easyanimate_b200 import EasyAnimateControlPipeline
    from easyanimate_b200.transformer3d import EasyAnimateTransformer3DModel
    A = on_cpu
    g = torch.Generator().manual_seed(13)
    lat = torch.randn(1, 16, LF, H // 8, W // 8, generator=g).to(bf16)
    control = torch.rand(1, 3, FRAMES, H, W, generator=g)
    ref_image = torch.rand(1, 3, 1, H, W, generator=g) if with_ref_image else None
    pe, ne = (torch.randn(1, 9, 128, generator=g) * 3).to(bf16), (torch.randn(1, 9, 128, generator=g) * 3).to(bf16)
    ocfg = {k: v for k, v in CONTROL_CFG.items() if k in CFG}
    ob = dit.init_weights_(dit.OracleTransformer3D(**ocfg), 61).to(bf16)
    ov = vae.init_weights_(vae.OracleAutoencoderKLMagvit(block_out_channels=list(BOC), with_encoder=True), 62).to(bf16)
    kw = dict(height=H, width=W, video_length=FRAMES, num_inference_steps=STEPS)

    def reference_call():
        from oracle import ref_dit, ref_vae
        rt = ref_dit.reference_transformer(**CONTROL_CFG).eval()
        rt.load_state_dict(ob.state_dict(), strict=True)
        rv = ref_vae.reference_autoencoder(block_out_channels=BOC).eval()
        rv.load_state_dict(ov.state_dict(), strict=True)
        return ref_pipeline.run_control(ref_pipeline.reference_control_pipeline(rt.to(bf16), rv.to(bf16)), lat, control, ref_image,
                                        pe, ne, **kw)

    want = refgold.want(f"ref_pipeline/control_reference_modules_{with_ref_image}", reference_call)
    ours_t = EasyAnimateTransformer3DModel(**CONTROL_CFG).to(bf16)
    ours_t.load_state_dict(ob.state_dict(), strict=True)
    ours_v = A.AutoencoderKLMagvit(latent_channels=16, cache_mag_vae=True, spatial_group_norm=True, mid_block_attention_type="spatial",
                                   block_out_channels=list(BOC), scaling_factor=0.7125, mini_batch_encoder=4,
                                   mini_batch_decoder=1).to(bf16)
    ours_v.load_state_dict(ov.state_dict(), strict=True)
    frames = ref_pipeline.run_control(EasyAnimateControlPipeline(vae=ours_v, transformer=ours_t), lat, control, ref_image, pe, ne,
                                      **kw)
    assert tuple(frames.shape) == want.shape == (1, 3, FRAMES, H, W) and frames.dtype == torch.float32
    rel = refgold.diff(frames, want)[1]
    assert rel < 3e-2, rel
