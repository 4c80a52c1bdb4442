"""CPU suite: the oracle against the golden vectors minted from the reference, against stored results of the reference run
on the same weights and inputs (tests/refgold.py), and internal consistency of the restated diffusers pieces."""
import ast
import os

import pytest
import torch
from safetensors import safe_open
from safetensors.torch import load_file

from oracle import dit, ref_dit, ref_vae, vae
from tests import refgold

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _meta(path):
    with safe_open(path, framework="pt") as f:
        return f.metadata()


@pytest.mark.parametrize("name", ["vae_small_attn", "vae_small_noattn_ragged", "vae_full_arch"])
def test_vae_oracle_matches_reference_golden(name):
    path = os.path.join(GOLD, f"{name}.safetensors")
    t, meta = load_file(path), _meta(path)
    boc = ast.literal_eval(meta["block_out_channels"])
    dec = vae.init_weights_(vae.OracleDecoder(block_out_channels=boc, mid_block_use_attention=meta["mid_attention"] == "True"),
                            int(meta["seed"]))
    with torch.no_grad():
        out = dec(t["z"])
    assert out.shape == t["out"].shape
    torch.testing.assert_close(out, t["out"], rtol=1e-4, atol=1e-4)  # whole-sequence vs chunked fp32 round-off


@pytest.mark.parametrize("cache", [True, False])
def test_vae_oracle_matches_live_reference(cache):
    boc = (64, 64, 128, 128)
    mine = vae.init_weights_(vae.OracleDecoder(block_out_channels=boc), 3)
    z = torch.randn(1, 16, 3, 6, 8, generator=torch.Generator().manual_seed(5))

    def reference_call():
        ref = ref_vae.reference_decoder(cache_mag_vae=cache, block_out_channels=boc)
        ref.load_state_dict(mine.state_dict(), strict=True)
        with torch.no_grad():
            return ref(z)

    want = refgold.want(f"oracle/vae_decoder_cache_{cache}", reference_call)
    with torch.no_grad():
        refgold.assert_close(mine(z), want, rtol=1e-4, atol=1e-4)


def test_vae_oracle_wrapper_matches_reference_golden():
    """decode / tiled_decode of the REFERENCE's AutoencoderKLMagvit wrapper (post_quant_conv, 3 x 3 tiles + the
    lower-right corner pass, blend_v / blend_h order): tests/golden/make_golden.py::make_vae_tiled."""
    path = os.path.join(GOLD, "vae_ref_tiled.safetensors")
    t, meta = load_file(path), _meta(path)
    boc = ast.literal_eval(meta["block_out_channels"])
    m = vae.init_weights_(vae.OracleAutoencoderKLMagvit(block_out_channels=boc, use_tiling=True,
                                                        tile_sample_min_size=int(meta["tile_sample_min_size"])), int(meta["seed"]))
    with torch.no_grad():
        tiled = m.decode(t["z"])[0]
        m.use_tiling = False
        full = m.decode(t["z"])[0]
    torch.testing.assert_close(tiled, t["out_tiled"], rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(full, t["out_untiled"], rtol=1e-4, atol=1e-4)


def test_vae_oracle_wrapper_matches_live_reference():
    boc = (64, 64, 128, 128)
    mine = vae.init_weights_(vae.OracleAutoencoderKLMagvit(block_out_channels=boc, use_tiling=True, tile_sample_min_size=64), 9)
    z = torch.randn(1, 16, 2, 12, 20, generator=torch.Generator().manual_seed(1))

    def reference_call():
        ref = ref_vae.reference_autoencoder(block_out_channels=boc, use_tiling=True, tile_sample_min_size=64)
        missing, unexpected = ref.load_state_dict(mine.state_dict(), strict=False)
        with torch.no_grad():
            return {"missing": list(missing), "unexpected": list(unexpected), "out": ref.decode(z).sample}

    want = refgold.want("oracle/vae_wrapper_tiled", reference_call)
    assert not want["unexpected"] and all(k.startswith(("encoder.", "quant_conv.")) for k in want["missing"])
    with torch.no_grad():
        refgold.assert_close(mine.decode(z)[0], want["out"], rtol=1e-4, atol=1e-4)


def test_vae_oracle_encode_matches_reference_golden():
    """encode / tiled_encode moments of the REFERENCE's AutoencoderKLMagvit (chunked Encoder: frame 0 alone, then four
    frames at a time with cached context): the whole-sequence encoder oracle reproduces them (I2V conditioning prep,
    SURVEY.md section 8(f) 'next' row - no CUDA path yet)."""
    path = os.path.join(GOLD, "vae_ref_encode.safetensors")
    t, meta = load_file(path), _meta(path)
    boc = ast.literal_eval(meta["block_out_channels"])
    m = vae.init_weights_(vae.OracleAutoencoderKLMagvit(block_out_channels=boc, with_encoder=True), int(meta["seed"]))
    with torch.no_grad():
        torch.testing.assert_close(m.encode_moments(t["x"]), t["moments"], rtol=1e-4, atol=1e-4)
        m.use_tiling, m.tile_sample_min_size, m.tile_latent_min_size = True, 32, 4
        torch.testing.assert_close(m.encode_moments(t["x"]), t["moments_tiled32"], rtol=1e-4, atol=1e-4)


def test_vae_oracle_encode_matches_live_reference():
    boc = (64, 64, 128, 128)
    mine = vae.init_weights_(vae.OracleAutoencoderKLMagvit(block_out_channels=boc, with_encoder=True), 5)
    x = torch.randn(1, 3, 5, 24, 40, generator=torch.Generator().manual_seed(6))

    def reference_call():
        ref = ref_vae.reference_autoencoder(block_out_channels=boc, use_tiling=False)
        ref.load_state_dict(mine.state_dict(), strict=True)  # all 244 keys, encoder included
        with torch.no_grad():
            return {"keys": sorted(ref.state_dict()), "moments": ref.encode(x).latent_dist.parameters}

    want = refgold.want("oracle/vae_encode", reference_call)
    assert sorted(mine.state_dict()) == want["keys"] and len(want["keys"]) == 244
    with torch.no_grad():
        refgold.assert_close(mine.encode_moments(x), want["moments"], rtol=1e-4, atol=1e-4)


def test_vae_tiled_decode_oracle_shapes_and_seams():
    m = vae.init_weights_(vae.OracleAutoencoderKLMagvit(block_out_channels=(64, 64, 128, 128), use_tiling=True,
                                                        tile_sample_min_size=64, mid_block_use_attention=False), 9)
    z = torch.randn(1, 16, 2, 12, 20, generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        tiled = m.decode(z)[0]
        m.use_tiling = False
        full = m.decode(z)[0]
    assert tiled.shape == full.shape == (1, 3, 5, 96, 160)
    assert torch.isfinite(tiled).all()


def _dit_case(name):
    path = os.path.join(GOLD, f"{name}.safetensors")
    t, meta = load_file(path), _meta(path)
    cfg = ast.literal_eval(meta["config"])
    m = dit.init_weights_(dit.OracleTransformer3D(**cfg), int(meta["seed"])).eval()
    return t, meta, cfg, m


@pytest.mark.parametrize("name", ["dit_ref_t2v", "dit_ref_i2v_inpaint", "dit_ref_3heads_3layers"])
def test_dit_oracle_matches_reference_golden(name):
    """Outputs of the REFERENCE's EasyAnimateTransformer3DModel (tests/golden/make_golden.py::make_dit_reference)."""
    t, meta, cfg, m = _dit_case(name)
    B, F, H, W, St = ast.literal_eval(meta["shape"])
    rope = dit.rope_for_video(H * 8, W * 8, F)
    with torch.no_grad():
        out = m(t["latents"], t["timestep"], encoder_hidden_states=t["encoder_hidden_states"], image_rotary_emb=rope,
                inpaint_latents=t.get("inpaint_latents"))[0]
    torch.testing.assert_close(out, t["out"], rtol=1e-5, atol=1e-6)


def test_dit_oracle_control_ref_clip_matches_reference_golden():
    """The Control model's reference-image / CLIP token branches (transformer3d.py:1420-1429,1538-1561), fixture minted by
    the reference module; the 2-D sin-cos table is diffusers' (restated, unpinned) in oracle and shim alike."""
    t, meta, cfg, m = _dit_case("dit_ref_control_ref_clip")
    m = m.to(torch.float32)  # the float64 position-table buffer follows the module dtype, like under .to(bfloat16)
    rope = dit.rope_for_video(64, 96, 2)
    kw = dict(encoder_hidden_states=t["encoder_hidden_states"], image_rotary_emb=rope, ref_latents=t["ref_latents"])
    with torch.no_grad():
        out = m(t["latents"], t["timestep"], clip_encoder_hidden_states=t["clip_encoder_hidden_states"], **kw)[0]
        out_ref_only = m(t["latents"], t["timestep"], **kw)[0]
    torch.testing.assert_close(out, t["out"], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(out_ref_only, t["out_ref_only"], rtol=1e-5, atol=1e-6)
    assert not torch.allclose(out, out_ref_only, atol=1e-3)


def test_dit_oracle_teacache_matches_reference_golden():
    """Six calls of the reference model with TeaCache enabled: same skip decisions, same outputs."""
    t, meta, cfg, m = _dit_case("dit_ref_teacache")
    m.teacache = dit.OracleTeaCache(ast.literal_eval(meta["coefficients"]), int(meta["num_steps"]), float(meta["rel_l1_thresh"]))
    rope = dit.rope_for_video(64, 96, 3)
    skipped = []
    with torch.no_grad():
        for i in range(6):
            before = m.teacache.skipped
            out = m(t["latents"] * (1.0 - 0.01 * i), t["timestep"] - 30.0 * i, encoder_hidden_states=t["encoder_hidden_states"],
                    image_rotary_emb=rope)[0]
            skipped.append(float(m.teacache.skipped - before))
            torch.testing.assert_close(out, t["outs"][i], rtol=1e-5, atol=1e-6)
    assert skipped == t["skipped"].tolist() and sum(skipped) == 3


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_dit_oracle_matches_live_reference_bit_for_bit(dtype):
    """The reference's own transformer3d.py / attention.py / processor.py / norm.py, executed unmodified
    (oracle/ref_dit.py), against the restatement with the same weights: identical in fp32 and in bf16 (the op-by-op
    rounding points are the same) on the CPU configuration the reference's output was stored on; elsewhere within the spread
    the CPU instruction set and thread count cause (tests/refgold.py)."""
    cfg = dict(num_attention_heads=2, attention_head_dim=64, in_channels=16, out_channels=16, patch_size=2, num_layers=2,
               time_embed_dim=64, add_norm_text_encoder=True, text_embed_dim=128, text_embed_dim_t5=None)
    mine = dit.init_weights_(dit.OracleTransformer3D(**cfg), 7).eval()
    g = torch.Generator().manual_seed(1)
    lat = torch.randn(2, 16, 3, 8, 12, generator=g).to(dtype)
    enc = (torch.randn(2, 40, 128, generator=g) * 3).to(dtype)
    tt = torch.tensor([937.0, 421.0]).to(dtype)
    rope = dit.rope_for_video(64, 96, 3)

    def reference_call():
        ref = ref_dit.reference_transformer(**cfg).eval()
        ref.load_state_dict(mine.state_dict(), strict=True)
        with torch.no_grad():
            return ref.to(dtype)(lat, tt, encoder_hidden_states=enc, image_rotary_emb=rope, return_dict=False)[0]

    a = refgold.want(f"oracle/dit_{str(dtype).split('.')[-1]}", reference_call)
    mine = mine.to(dtype)
    with torch.no_grad():
        b = mine(lat, tt, encoder_hidden_states=enc, image_rotary_emb=rope)[0]
    refgold.assert_equal(b, a, rel=1e-5 if dtype == torch.float32 else 3e-2)


def test_dit_golden_regression():
    t = load_file(os.path.join(GOLD, "dit_tiny.safetensors"))
    from tests.golden.make_golden import DIT_CFG
    m = dit.init_weights_(dit.OracleTransformer3D(**DIT_CFG), 1234)
    rope = dit.rope_for_video(64, 96, 3)
    torch.testing.assert_close(rope[0], t["rope_cos"])
    torch.testing.assert_close(rope[1], t["rope_sin"])
    out = dit.denoise_loop(m, t["latents"], t["prompt_embeds"], t["negative_prompt_embeds"], rope, 3, 6.0)
    torch.testing.assert_close(out, t["out_3steps_cfg6"], rtol=1e-4, atol=1e-4)
    s = dit.FlowMatchEulerScheduler(shift=3.0)
    s.set_timesteps(25, mu=1.0)
    torch.testing.assert_close(s.sigmas, t["sigmas_shift3_25"])
    c, sn = dit.rope_for_video(720, 1280, 2)
    torch.testing.assert_close(c[:200], t["rope720_cos_head"])
    torch.testing.assert_close(sn[-200:], t["rope720_sin_tail"])


def test_rope_crop_region_matches_reference_function():
    """The RoPE grid's crop region (pipeline_easyanimate.py:82-97) is reference-owned code: its function is lifted out of
    the pipeline file by AST (the file itself imports the text encoders); its results (stored) are compared with the oracle's
    and the product's host-side restatements over every latent grid a 16-pixel-aligned video up to 1536 x 1536 can produce."""
    import ast as _ast
    from easyanimate_b200 import pipeline as prod
    grids = [(gh, gw) for gh in range(1, 97) for gw in range(1, 97)]

    def reference_call():
        src = open(os.path.join(ref_dit.REFERENCE_ROOT, "easyanimate", "pipeline", "pipeline_easyanimate.py")).read()
        fn = next(n for n in _ast.parse(src).body if isinstance(n, _ast.FunctionDef) and n.name == "get_resize_crop_region_for_grid")
        ns = {}
        exec(compile(_ast.Module(body=[fn], type_ignores=[]), "<reference>", "exec"), ns)
        return torch.tensor([ns["get_resize_crop_region_for_grid"](g, 45, 30) for g in grids])

    regions = refgold.want("oracle/rope_crop_regions", reference_call)
    assert regions.shape == (len(grids), 2, 2)
    for g, r in zip(grids, regions.values.reshape(regions.shape).tolist()):
        want = tuple(tuple(x) for x in r)
        assert dit.get_resize_crop_region_for_grid(g, 45, 30) == want
        assert prod.get_resize_crop_region_for_grid(g, 45, 30) == want


def test_rope_properties():
    cos, sin = dit.rope_for_video(720, 1280, 13)
    assert cos.shape == (13 * 45 * 80, 64) and cos.dtype == torch.float32
    torch.testing.assert_close(cos * cos + sin * sin, torch.ones_like(cos))
    # pairs are repeat-interleaved, and the temporal band (first 16 dims) is constant inside a frame
    assert torch.equal(cos[:, 0::2], cos[:, 1::2])
    assert torch.equal(cos[:45 * 80, :16], cos[0:1, :16].expand(45 * 80, 16))
    # rotating by the table is norm-preserving
    x = torch.randn(1, 2, 13 * 45 * 80, 64)
    y = dit.apply_rotary_emb(x, (cos, sin))
    torch.testing.assert_close(y.norm(dim=-1), x.norm(dim=-1), rtol=1e-4, atol=1e-4)


def test_scheduler_properties():
    for shift, dyn in ((1.0, False), (3.0, False), (1.0, True)):
        s = dit.FlowMatchEulerScheduler(shift=shift, use_dynamic_shifting=dyn)
        for n in (25, 30, 50):
            s.set_timesteps(n, mu=1.0)
            assert s.sigmas.shape == (n + 1,) and s.sigmas[-1] == 0
            assert torch.all(s.sigmas[:-1] > s.sigmas[1:])
            torch.testing.assert_close(s.timesteps, s.sigmas[:-1] * 1000)
    # Euler steps telescope: with a constant velocity v the loop integrates x0 + (0 - sigma_0) * v
    s = dit.FlowMatchEulerScheduler()
    s.set_timesteps(10)
    x, v = torch.zeros(4), torch.ones(4)
    for _ in range(10):
        x = s.step(v, x)
    torch.testing.assert_close(x, -s.sigmas[0] * torch.ones(4))


def test_cfg_linearity():
    """CFG with guidance g is linear in (u, c): g=1 returns c, g=0 returns u."""
    u, c = torch.randn(5), torch.randn(5)
    assert torch.allclose(u + 1.0 * (c - u), c)
    assert torch.allclose(u + 0.0 * (c - u), u)
