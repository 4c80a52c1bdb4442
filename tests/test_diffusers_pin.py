"""Pinning the third-party (`diffusers` 0.30.1-0.31.0) arithmetic the EasyAnimateV5.1 path calls, which oracle/dit.py and
oracle/_refshim restate because diffusers can be installed neither here nor on the GPU box (VERDICT round 1, weak item 4).

Part A compares the restatements with INDEPENDENT copies of the same published functions (results of the reference's copies
stored by tests/refgold.py; transformers' where it is installed):
  * `get_2d_sincos_pos_embed`  <- the reference's own vendored copy (easyanimate/models/patch.py:12-58, diffusers' function with
    interpolation_scale / base_size) and transformers' MAE original (models/vit_mae/modeling_vit_mae.py);
  * `get_timestep_embedding`   <- the reference's vendored DDPM original (easyanimate/vae/ldm/modules/diffusionmodules/model.py:
    12-32 = flip_sin_to_cos False, downscale_freq_shift 1), which fixes the exponent / (half_dim - shift) form and the sin|cos
    order that `flip_sin_to_cos=True, downscale_freq_shift=0` (transformer3d.py:1399, ctor defaults :1365,1377) then permutes;
  * GELU(tanh), SiLU, LayerNorm, scaled_dot_product_attention are torch's own kernels in diffusers too (nothing to restate).
Part B runs only where a real `diffusers` is importable (skipped otherwise - on both boxes of this build) and compares every
restated primitive with the real class / function: scheduler, 3-D RoPE table, Timesteps, apply_rotary_emb, AdaLayerNorm,
FeedForward(gelu-approximate), get_2d_sincos_pos_embed.  Until Part B has run somewhere, the scheduler and
`get_3d_rotary_pos_embed` stay "parity unpinned" (DESIGN.md section 4)."""
import ast
import importlib.util
import math
import os
import sys

import numpy as np
import pytest
import torch

from oracle import dit, ref_dit
from tests import refgold

HERE = os.path.dirname(os.path.abspath(__file__))
SHIM_DIR = os.path.join(os.path.dirname(HERE), "oracle", "_refshim", "diffusers")
REF = ref_dit.REFERENCE_ROOT


def _shim():
    """oracle/_refshim/diffusers loaded under an alias, so that it can sit next to a real `diffusers`."""
    name = "_ea_diffusers_shim"
    if name not in sys.modules:
        spec = importlib.util.spec_from_file_location(name, os.path.join(SHIM_DIR, "__init__.py"),
                                                      submodule_search_locations=[SHIM_DIR])
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
    return importlib.import_module(name + ".models.embeddings"), importlib.import_module(name + ".schedulers")


def _lift(path, names, env):
    """Execute only the named top-level functions of a reference file (its module-level imports need packages this box lacks)."""
    tree = ast.parse(open(path).read())
    body = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in names]
    assert {n.name for n in body} == set(names), (path, names)
    ns = dict(env)
    exec(compile(ast.Module(body=body, type_ignores=[]), path, "exec"), ns)
    return ns


# ---- Part A ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dim,grid,base", [(128, (4, 6), 16), (256, (8, 8), 8), (64, (5, 3), 16)])
def test_sincos_2d_table_matches_the_references_vendored_copy(dim, grid, base):
    emb, _ = _shim()

    def reference_call():
        ref = _lift(os.path.join(REF, "easyanimate", "models", "patch.py"),
                    ["get_2d_sincos_pos_embed", "get_2d_sincos_pos_embed_from_grid", "get_1d_sincos_pos_embed_from_grid"], {"np": np})
        return ref["get_2d_sincos_pos_embed"](dim, grid, base_size=base)

    want = refgold.want(f"diffusers_pin/sincos_2d_{dim}_{grid[0]}x{grid[1]}_{base}", reference_call)
    got_shim = emb.get_2d_sincos_pos_embed(dim, grid, base_size=base)
    got_oracle = dit.sincos_pos_embed_2d(dim, grid, base_size=base)
    refgold.assert_equal(np.asarray(got_shim), want, rel=1e-12)
    got_oracle = np.asarray(got_oracle.numpy() if torch.is_tensor(got_oracle) else got_oracle).reshape(want.shape)
    refgold.assert_equal(got_oracle, want, rel=1e-12)


def test_sincos_2d_table_matches_transformers_mae_original():
    mae = pytest.importorskip("transformers.models.vit_mae.modeling_vit_mae")
    emb, _ = _shim()
    for dim, g in ((128, 6), (64, 9)):
        want = mae.get_2d_sincos_pos_embed(dim, g, add_cls_token=False)
        got = emb.get_2d_sincos_pos_embed(dim, g, base_size=g)  # base_size == grid_size: positions 0..g-1, MAE's own grid
        assert np.allclose(np.asarray(got), np.asarray(want), rtol=0, atol=1e-12)


@pytest.mark.parametrize("dim", [64, 128, 512])
def test_timestep_embedding_matches_the_references_vendored_ddpm_original(dim):
    emb, _ = _shim()
    t = torch.tensor([0.0, 1.0, 421.0, 937.5, 1000.0])

    def reference_call():
        ref = _lift(os.path.join(REF, "easyanimate", "vae", "ldm", "modules", "diffusionmodules", "model.py"),
                    ["get_timestep_embedding"], {"math": math, "torch": torch})
        return ref["get_timestep_embedding"](t, dim)

    want = refgold.want(f"diffusers_pin/timestep_embedding_{dim}", reference_call)
    for f in (emb.get_timestep_embedding, dit.get_timestep_embedding):
        # same formula, different association of the fp32 products (DDPM: arange * (-log/(h-1)); diffusers: (-log * arange)/(h-1)):
        # arguments up to 1000 rad -> 1e-7 relative is ~1e-4 absolute in sin / cos
        refgold.assert_close(f(t, dim, flip_sin_to_cos=False, downscale_freq_shift=1), want, rtol=0, atol=3e-4)
        # the EasyAnimate configuration (transformer3d.py:1399 Timesteps(inner_dim, flip_sin_to_cos=True, freq_shift=0)): cos | sin, exponent / half_dim
        half = dim // 2
        freqs = torch.exp(-math.log(10000) * torch.arange(half, dtype=torch.float32) / half)
        arg = t[:, None].float() * freqs[None]
        assert torch.equal(f(t, dim, flip_sin_to_cos=True, downscale_freq_shift=0), torch.cat([arg.cos(), arg.sin()], dim=-1))


def test_oracle_and_shim_restatements_agree_with_each_other():
    """Two restatements written separately (oracle/dit.py for the oracle, oracle/_refshim for the reference's imports)."""
    emb, sch = _shim()
    x = torch.randn(2, 3, 10, 64, generator=torch.Generator().manual_seed(0))
    rope = dit.rope_for_video(32, 80, 1)
    assert torch.equal(emb.apply_rotary_emb(x, rope), dit.apply_rotary_emb(x, rope))
    a, b = sch.FlowMatchEulerDiscreteScheduler(shift=3.0), dit.FlowMatchEulerScheduler(shift=3.0)
    a.set_timesteps(7, device="cpu", mu=1)
    b.set_timesteps(7, mu=1)
    assert torch.equal(a.timesteps, b.timesteps) and torch.equal(a.sigmas, b.sigmas)
    v, s = torch.randn(4, 5).to(torch.bfloat16), torch.randn(4, 5).to(torch.bfloat16)
    assert torch.equal(a.step(v, a.timesteps[0], s, return_dict=False)[0], b.step(v, s))


# ---- Part B: against a real diffusers, wherever one is importable --------------------------------------------------------
def _real_diffusers():
    for extra in (os.path.join(os.path.dirname(HERE), "baseline", "_ref"),):
        if os.path.isdir(extra) and extra not in sys.path:
            sys.path.append(extra)
    d = pytest.importorskip("diffusers")
    if os.path.abspath(os.path.dirname(d.__file__)) == os.path.abspath(SHIM_DIR):
        pytest.skip("only the oracle's stand-in is importable as `diffusers` here")
    return d


def test_real_diffusers_scheduler():
    _real_diffusers()
    from diffusers.schedulers import FlowMatchEulerDiscreteScheduler as Real
    from easyanimate_b200.scheduler import FlowMatchEulerDiscreteScheduler as Ours
    _, sch = _shim()
    for shift, n in ((1.0, 30), (3.0, 50), (1.0, 1)):
        real, shim, ours, orc = Real(shift=shift), sch.FlowMatchEulerDiscreteScheduler(shift=shift), Ours(shift=shift), \
            dit.FlowMatchEulerScheduler(shift=shift)
        real.set_timesteps(n, device="cpu")
        shim.set_timesteps(n, device="cpu")
        ours.set_timesteps(n, device="cpu")
        orc.set_timesteps(n)
        for other in (shim, ours, orc):
            assert torch.equal(real.timesteps, torch.as_tensor(other.timesteps)) and torch.equal(real.sigmas, torch.as_tensor(other.sigmas))
        v, s = torch.randn(3, 7).to(torch.bfloat16), torch.randn(3, 7).to(torch.bfloat16)
        want = real.step(v, real.timesteps[0], s, return_dict=False)[0]
        assert torch.equal(want, shim.step(v, shim.timesteps[0], s, return_dict=False)[0])
        assert torch.equal(want, orc.step(v, s))


def test_real_diffusers_embeddings_and_layers():
    _real_diffusers()
    from diffusers.models import embeddings as R
    emb, _ = _shim()
    crops = dit.get_resize_crop_region_for_grid((45, 80), 45, 30)
    want = R.get_3d_rotary_pos_embed(64, crops, grid_size=(45, 80), temporal_size=13, use_real=True)
    got = dit.get_3d_rotary_pos_embed(64, crops, (45, 80), 13)
    assert torch.equal(want[0], got[0]) and torch.equal(want[1], got[1])
    t = torch.tensor([0.0, 421.0, 937.5])
    for f in (emb.get_timestep_embedding, dit.get_timestep_embedding):
        assert torch.equal(R.get_timestep_embedding(t, 512, flip_sin_to_cos=True, downscale_freq_shift=0),
                           f(t, 512, flip_sin_to_cos=True, downscale_freq_shift=0))
    x = torch.randn(2, 3, 13 * 45 * 80 // 100, 64)
    rope = (want[0][: x.shape[2]], want[1][: x.shape[2]])
    assert torch.equal(R.apply_rotary_emb(x, rope), dit.apply_rotary_emb(x, rope))
    assert np.array_equal(np.asarray(R.get_2d_sincos_pos_embed(128, (4, 6))), np.asarray(emb.get_2d_sincos_pos_embed(128, (4, 6))))
    from diffusers.models.attention import FeedForward
    from diffusers.models.normalization import AdaLayerNorm
    g = torch.Generator().manual_seed(1)
    ff_r, ff_o = FeedForward(64, dropout=0.0, activation_fn="gelu-approximate", final_dropout=True, inner_dim=256, bias=True), \
        dit.FeedForward(64, 256)
    ff_o.load_state_dict(ff_r.state_dict())
    h = torch.randn(2, 5, 64, generator=g)
    assert torch.equal(ff_r(h), ff_o(h))
    ad_r, ad_o = AdaLayerNorm(embedding_dim=32, output_dim=128, norm_elementwise_affine=True, norm_eps=1e-5, chunk_dim=1), \
        dit.AdaLayerNorm(32, 128, 1e-5)
    ad_o.load_state_dict(ad_r.state_dict())
    temb = torch.randn(2, 32, generator=g)
    assert torch.equal(ad_r(h, temb=temb), ad_o(h, temb))
