#!/usr/bin/env python
"""bench.py — EasyAnimateV5.1 sampling hot path on B200 (BASELINE.json metric: denoising-steps/sec @49f·720p bf16).

    python bench.py --gpus N --steps K --warmup W            # our arm (torchrun launches one rank per GPU for N>1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU path (oracle port), rank 0 only

A "step" is ONE scheduler step of the denoise loop WITH classifier-free guidance: two MMDiT forwards (batch of 2), the
CFG combine and the flow-matching Euler update (pipeline_easyanimate.py:1069-1111).  Workload at N=1: BASELINE
configs[1] read as SURVEY.md §8(d) resolves it — "7B" synthetic MMDiT (d=3072, 48 heads, 28 layers, 6.87 B params),
49 frames @720x1280 => latent 13x90x160 => 46 800 video + 256 text tokens, synthetic text embeds, random-init weights.

Topology for N > 1 (one process per GPU): N = 2 -> the two CFG branches on one GPU each (one 6 MB all_gather per step);
N >= 4 -> still ONE video: 2 CFG branches x N/2 sequence-parallel ranks (easyanimate_b200/sequence_parallel.py), so the
N = 1..8 sweep is STRONG scaling of one video's step.  EA_BENCH_TOPOLOGY=replicas restores independent videos per pair.

Besides the headline line the JSON carries (rank 0): `roofline` of the dominant kernel, `e2e` with host buffers, `secondary`
lines for the other BASELINE configs that fit the run (12B, I2V 1024^2 12B with vae.encode, VAE decode untiled / tiled /
to-host with its own roofline), `torch_gpu_baseline` (the oracle's stock-PyTorch modules - cuBLAS, cuDNN/flash SDPA - on the
same GPU, same config) and `cpu_baseline` (oracle port on the host cores, bounded sample).  Prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PRESETS = {
    # name: latent F,h,w, layers, heads (+ inpaint: 17 conditioning channels concatenated, in_channels 33)
    "R720_7B": dict(F=13, h=90, w=160, layers=28, heads=48),
    "R720_12B": dict(F=13, h=90, w=160, layers=48, heads=48),
    "R512_7B": dict(F=13, h=64, w=64, layers=28, heads=48),
    "R1024_12B_I2V": dict(F=13, h=128, w=128, layers=48, heads=48, inpaint=True),
    "tiny": dict(F=3, h=16, w=24, layers=2, heads=4),
    "tiny_I2V": dict(F=3, h=16, w=24, layers=2, heads=4, inpaint=True),
}
S_TEXT, E_TEXT, GUIDANCE = 256, 3584, 6.0
METRIC = "denoising-steps/sec @49f·720p bf16 (CFG step = 2 MMDiT forwards)"
_CPU_THREADS = None


def dit_flops_per_forward(F, h, w, layers, heads, c_in=16, s_t=S_TEXT, e_text=E_TEXT, inpaint=False):
    """BASELINE.md §2 closed form (MAC = 2 FLOP; softmax/LN/GELU excluded)."""
    d = heads * 64
    s_v = F * (h // 2) * (w // 2)
    s = s_v + s_t
    c_in = 33 if inpaint else c_in
    return layers * (24 * s * d * d + 4 * s * s * d) + 2 * s_v * 4 * c_in * d + 2 * s_t * e_text * d + 2 * s_v * d * 64


def model_cfg(p, text_dim=E_TEXT):
    return dict(num_attention_heads=p["heads"], attention_head_dim=64, in_channels=33 if p.get("inpaint") else 16,
                out_channels=16, patch_size=2, num_layers=p["layers"], time_embed_dim=512, add_norm_text_encoder=True,
                text_embed_dim=text_dim, text_embed_dim_t5=None)


def _flop_args(p):
    return {k: p[k] for k in ("F", "h", "w", "layers", "heads")} | ({"inpaint": True} if p.get("inpaint") else {})


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w": statistics.median(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
# CPU legs (the only places that import oracle/)
# ---------------------------------------------------------------------------------------------------------------
CPU_SAMPLE = dict(F=1, h=64, w=64, layers=1, heads=48)  # 1 024 video + 256 text tokens, one MMDiT block of the real width


def cpu_oracle_rate(seconds_budget: float = 15.0, threads: int | None = None, min_reps: int = 2):
    """Reference CPU path = the oracle restatement (diffusers is not installable offline, DESIGN.md): one
    EasyAnimateDiTBlock-deep model (d=3072, 48 heads) on 1 024 video + 256 text tokens, CFG batch 2, bf16, all host
    cores.  Returns (flop/s, description, cores, per-rep seconds list)."""
    import torch
    from oracle import dit
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    p = CPU_SAMPLE
    if threads is None:
        # "all the host threads it can use": torch's bf16 CPU kernels stop scaling (and regress badly) well before 128
        # threads on this small sample, so probe a few team sizes once and keep the fastest.
        global _CPU_THREADS
        if _CPU_THREADS is None:
            best = (float("inf"), avail)
            probe = dit.OracleTransformer3D(**model_cfg(dict(p, heads=8))).to(torch.bfloat16)
            x = torch.randn(2, 16, 1, 32, 32).to(torch.bfloat16)
            e = torch.randn(2, 64, E_TEXT).to(torch.bfloat16)
            rp = dit.rope_for_video(256, 256, 1)
            tt = torch.tensor([500.0, 500.0]).to(torch.bfloat16)
            for n in sorted({avail, max(1, avail // 2), max(1, avail // 4), min(avail, 32), min(avail, 16), min(avail, 8)}):
                torch.set_num_threads(n)
                with torch.no_grad():
                    probe(x, tt, encoder_hidden_states=e, image_rotary_emb=rp)
                    t0 = time.perf_counter()
                    probe(x, tt, encoder_hidden_states=e, image_rotary_emb=rp)
                    dt = time.perf_counter() - t0
                if dt < best[0]:
                    best = (dt, n)
            _CPU_THREADS = best[1]
        threads = _CPU_THREADS
    torch.set_num_threads(threads)
    m = dit.OracleTransformer3D(**model_cfg(p)).to(torch.bfloat16)
    g = torch.Generator().manual_seed(0)
    lat = torch.randn(2, 16, p["F"], p["h"], p["w"], generator=g).to(torch.bfloat16)
    enc = torch.randn(2, S_TEXT, E_TEXT, generator=g).to(torch.bfloat16)
    rope = dit.rope_for_video(p["h"] * 8, p["w"] * 8, p["F"])
    t = torch.tensor([500.0, 500.0]).to(torch.bfloat16)
    fl = 2 * dit_flops_per_forward(**p)
    times = []
    with torch.no_grad():
        m(lat, t, encoder_hidden_states=enc, image_rotary_emb=rope)  # warm-up
        t_end = time.perf_counter() + seconds_budget
        while time.perf_counter() < t_end or len(times) < min_reps:
            t0 = time.perf_counter()
            m(lat, t, encoder_hidden_states=enc, image_rotary_emb=rope)
            times.append(time.perf_counter() - t0)
    per = statistics.median(times)
    desc = (f"oracle/dit.py (torch-cpu bf16, {threads} of {avail} available threads — fastest team size probed): 1 MMDiT block "
            f"d=3072/48 heads, CFG batch 2, 1024 video + 256 text tokens, {len(times)} reps, median {per:.3f} s/rep; steps/s "
            f"extrapolated by FLOPs to the workload")
    return fl / per, desc, threads, times


def run_reference_arm(args, preset):
    """--impl reference: the reference's own CPU implementation of the path on the host cores (oracle port).  One "step" of
    this arm is ONE timed evaluation of the bounded sample (CPU_SAMPLE: one MMDiT block of the real width on 1 280 tokens,
    CFG batch 2); `ms_per_step` is that measured time, `value` the workload's steps/s extrapolated from it by FLOP count -
    a full R720 step is ~5.5 hours of this CPU path, so it cannot be run; the line says so (`extrapolated`)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    flops_step = 2 * dit_flops_per_forward(**_flop_args(preset))
    flops_sample = 2 * dit_flops_per_forward(**CPU_SAMPLE)
    _, desc, cores, _ = cpu_oracle_rate(seconds_budget=0.0, min_reps=max(1, args.warmup))     # warm-up reps
    _, desc, cores, times = cpu_oracle_rate(seconds_budget=0.0, min_reps=max(1, args.steps))  # the timed "steps"
    ms_sample = statistics.mean(times[-args.steps:]) * 1e3
    rate = flops_sample / (ms_sample * 1e-3)
    value = rate / flops_step
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_sample, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic", "extrapolated": True,
            "extrapolation": {"measured": "ms_per_step = one evaluation of the bounded sample", "sample_tflop": flops_sample / 1e12,
                              "workload_tflop_per_step": flops_step / 1e12, "cpu_tflops": rate / 1e12,
                              "ms_per_workload_step_extrapolated": flops_step / rate * 1e3},
            "config": {"workload": args.preset, **{k: v for k, v in preset.items()}},
            "cpu_baseline": {"value": value, "unit": "steps/s", "cores": cores, "kind": "port", "sample": desc},
            "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------
# helpers of our arm
# ---------------------------------------------------------------------------------------------------------------
def build_model(preset, dev, seed=1234):
    import torch
    from easyanimate_b200.transformer3d import EasyAnimateTransformer3DModel
    torch.manual_seed(seed)  # identical weights on every rank
    with torch.device(dev):
        model = EasyAnimateTransformer3DModel(**model_cfg(preset)).to(torch.bfloat16)
    with torch.no_grad():
        for name, prm in model.named_parameters():
            if prm.dim() == 1 and name.endswith("weight"):
                prm.normal_(1.0, 0.02)
            else:
                prm.normal_(0.0, 0.02)
    return model


def build_vae(dev, tiled=False):
    import torch
    from easyanimate_b200.autoencoder_magvit import AutoencoderKLMagvit
    with torch.device(dev):
        vae = AutoencoderKLMagvit(latent_channels=16, cache_mag_vae=True, spatial_group_norm=True,
                                  mid_block_attention_type="spatial", mini_batch_decoder=1, mini_batch_encoder=4,
                                  scaling_factor=0.7125, use_tiling=tiled).to(torch.bfloat16)
    with torch.no_grad():
        for n, p in vae.named_parameters():
            if p.dim() >= 2:
                p.normal_(0, (1.0 / p[0].numel()) ** 0.5)
            elif "norm" in n and n.endswith("weight"):
                p.normal_(1.0, 0.05)
            else:
                p.normal_(0, 0.05)
    return vae


def vae_decode_work(vae, F, h, w):
    """Algorithmic work of AutoencoderKLMagvit.decode for a [1,16,F,h,w] latent, walked over the module structure
    (SURVEY.md §8d: conv FLOPs = sum 2*(T*H*W)_out*C_out*27*C_in, 1x1x1 without the 27; bytes = each conv's input + output
    once in bf16).  Returns (conv_flops, attn_flops, bytes)."""
    fl, by, at = 0, 0, 0
    dec = vae.decoder

    def conv(c, T, H, W, cin=None, k=27):
        nonlocal fl, by
        cin = cin or c.in_channels
        fl += 2 * T * H * W * c.out_channels * k * cin
        by += 2 * T * H * W * (cin + c.out_channels)

    def res(r, T, H, W):
        conv(r.conv1, T, H, W); conv(r.conv2, T, H, W)
        if not isinstance(r.shortcut, __import__("torch").nn.Identity):
            conv(r.shortcut, T, H, W, k=1)

    T, H, W = F, h, w
    conv(vae.post_quant_conv, T, H, W, k=1)
    conv(dec.conv_in, T, H, W)
    res(dec.mid_block.convs[0], T, H, W)
    for a, r in zip(dec.mid_block.attentions, dec.mid_block.convs[1:]):
        if a is not None:
            Cc = a.to_q.in_features
            fl += 4 * 2 * T * H * W * Cc * Cc            # q, k, v, out projections
            at += 4 * T * (H * W) * (H * W) * Cc          # QK^T and PV per frame
        res(r, T, H, W)
    for up in dec.up_blocks:
        for r in up.convs:
            res(r, T, H, W)
        if up.upsampler is not None:
            H, W = 2 * H, 2 * W
            conv(up.upsampler.conv, T, H, W)
            if up.upsampler.temporal and T > 1:
                T = 2 * T - 1
    conv(dec.conv_out, T, H, W)
    return fl, at, by, (T, H, W)


def time_cuda(fn, reps, warmup=1):
    import torch
    for _ in range(warmup):
        out = fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return statistics.median(ts), out


def vae_lines(preset, dev, peaks, reps=3):
    """Secondary metric of the path (BASELINE.json: "VAE decode MPix/s"; configs[3]): AutoencoderKLMagvit.decode of the
    workload's latent - untiled whole-sequence, reference-faithful tiled (use_tiling, 384-px tiles, 16 decoder passes at
    720p, autoencoder_magvit.py:381-448), and end to end (latents from pinned host memory, 1/scaling_factor, decode, clamp,
    float32 frames stored into pinned host memory = pipeline_easyanimate.py:722-742) - each with its roofline."""
    import torch
    bf16 = torch.bfloat16
    vae = build_vae(dev)
    F, h, w = preset["F"], preset["h"], preset["w"]
    z = (torch.randn((1, 16, F, h, w), device=dev) / 0.7125).to(bf16)
    conv_fl, attn_fl, nbytes, (T, H, W) = vae_decode_work(vae, F, h, w)
    mpix = T * H * W / 1e6
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_bw = peaks.get("hbm_gbs", 6650.0)
    out = {}
    ms, y = time_cuda(lambda: vae.decode(z).sample, reps)
    out["untiled"] = {"value": mpix / ms * 1e3, "unit": "MPix/s", "ms": ms, "frames": T, "resolution": [H, W],
                      "mode": "untiled whole-sequence decode, random-init weights", "finite": bool(torch.isfinite(y).all()),
                      "roofline": {"bound": "tensor", "achieved": (conv_fl + attn_fl) / ms / 1e9, "peak": peak_tf, "unit": "TFLOP/s",
                                   "frac": (conv_fl + attn_fl) / ms / 1e9 / peak_tf, "conv_tflop": conv_fl / 1e12,
                                   "attn_tflop": attn_fl / 1e12, "algorithmic_gb": nbytes / 1e9,
                                   "hbm_gbs_algorithmic": nbytes / ms / 1e6, "hbm_frac": nbytes / ms / 1e6 / peak_bw,
                                   "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained / hbm_gbs (of measured)" if peaks else "fallback"}}
    del y
    # end to end with host buffers
    z_host = torch.empty(z.shape, dtype=bf16, pin_memory=True).copy_(z * 0.7125)
    frames = torch.empty((1, 3, T, H, W), dtype=torch.float32, pin_memory=True)

    def e2e():
        zz = z_host.to(dev, non_blocking=True)
        return vae.decode_scaled(zz, out=frames)
    ms_e, _ = time_cuda(e2e, max(2, reps - 1))
    out["e2e"] = {"value": mpix / ms_e * 1e3, "unit": "MPix/s", "ms": ms_e, "h2d_bytes": z_host.numel() * 2,
                  "d2h_bytes": frames.numel() * 4,
                  "mode": "decode_latents: latents from pinned host, 1/scaling_factor, decode, clamp, float32 frames written to "
                          "pinned host memory by the output kernel"}
    del frames
    vae.use_tiling = True
    ms_t, _ = time_cuda(lambda: vae.decode(z).sample, 2)
    tl = vae.tile_latent_min_size
    ov = int(tl * (1 - vae.tile_overlap_factor))
    passes = len(range(0, h, ov)) * len(range(0, w, ov)) + 1
    out["tiled"] = {"value": mpix / ms_t * 1e3, "unit": "MPix/s", "ms": ms_t, "decoder_passes": passes,
                    "mode": f"reference tiling: {tl}x{tl} latent tiles, stride {ov}, blend + corner pass (BASELINE configs[3])"}
    vae.use_tiling = False
    return out, vae


def torch_gpu_baseline(preset, dev, steps=2, warmup=1, with_vae=True):
    """The in-box baseline SURVEY.md §8(d) asks for: the SAME config and step through stock PyTorch on this GPU - the
    oracle's modules (nn.Linear -> cuBLAS, F.scaled_dot_product_attention -> flash/cuDNN, LayerNorm/GELU eager kernels),
    i.e. what the reference executes when handed a B200.  Baseline leg: never the product path."""
    import torch
    from oracle import dit
    bf16 = torch.bfloat16
    res = {}
    try:
        torch.manual_seed(7)
        with torch.device(dev):
            m = dit.OracleTransformer3D(**model_cfg(preset)).to(bf16)
        with torch.no_grad():
            for name, prm in m.named_parameters():
                prm.normal_(1.0 if (prm.dim() == 1 and name.endswith("weight")) else 0.0, 0.02)
        F, h, w = preset["F"], preset["h"], preset["w"]
        lat = torch.randn((1, 16, F, h, w), device=dev).to(bf16)
        emb = (torch.randn((2, S_TEXT, E_TEXT), device=dev) * 10).to(bf16)
        rope = tuple(t.to(dev) for t in dit.rope_for_video(h * 8, w * 8, F))
        sched = dit.FlowMatchEulerScheduler()
        sched.set_timesteps(max(30, steps + warmup + 1), mu=1.0)

        def step(lat, i):
            with torch.no_grad():
                x = torch.cat([lat] * 2)
                t = torch.tensor([float(sched.timesteps[i])] * 2, device=dev).to(bf16)
                pred = m(x, t, encoder_hidden_states=emb, image_rotary_emb=rope)[0]
                u, c = pred.chunk(2)
                pred = u + GUIDANCE * (c - u)
                sched.step_index = i
                return sched.step(pred, lat)
        i = 0
        for _ in range(warmup):
            lat = step(lat, i); i += 1
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            lat = step(lat, i); i += 1
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        res = {"value": 1e3 / ms, "unit": "steps/s", "ms_per_step": ms, "steps": steps, "warmup": warmup,
               "impl": f"oracle/dit.py modules on cuda, torch {torch.__version__} eager: cuBLAS linears, F.scaled_dot_product_attention, "
                       "eager LayerNorm/GELU/RoPE (what the reference's modules execute on a B200)",
               "model_tflops": 2 * dit_flops_per_forward(**_flop_args(preset)) / ms / 1e9, "finite": bool(torch.isfinite(lat).all())}
        del m, lat, emb
        torch.cuda.empty_cache()
    except Exception as e:  # a baseline that cannot run (e.g. out of memory in eager mode) must not take the bench down
        res = {"unavailable": f"{type(e).__name__}: {str(e)[:200]}"}
        torch.cuda.empty_cache()
    if with_vae:
        try:
            from oracle import vae as ovae
            with torch.device(dev):
                v = ovae.OracleAutoencoderKLMagvit(use_tiling=True).to(bf16)
            ovae.init_weights_(v, 3)
            F, h, w = preset["F"], preset["h"], preset["w"]
            tl = v.tile_latent_min_size
            z = torch.randn((1, 16, F, min(h, tl), min(w, tl)), device=dev).to(bf16)
            with torch.no_grad():
                v.decoder(v.post_quant_conv(z))
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                y = v.decoder(v.post_quant_conv(z))
                e1.record()
                torch.cuda.synchronize()
            ms_tile = e0.elapsed_time(e1)
            ov = int(tl * 0.75)
            passes = len(range(0, h, ov)) * len(range(0, w, ov)) + 1
            T, H, W = y.shape[2], 8 * h, 8 * w
            res["vae_decode_tiled"] = {"value": T * H * W / 1e6 / (ms_tile * passes) * 1e3, "unit": "MPix/s", "ms_per_tile": ms_tile,
                                       "decoder_passes": passes, "impl": "oracle/vae.py Decoder on cuda (F.conv3d -> cuDNN, whole-sequence "
                                       "form), ONE 48x48-latent tile timed, x passes of the reference tiling (blend excluded)"}
            del v, z, y
            torch.cuda.empty_cache()
        except Exception as e:
            res["vae_decode_tiled"] = {"unavailable": f"{type(e).__name__}: {str(e)[:200]}"}
            torch.cuda.empty_cache()
    return res


def load_traffic(kernel: str, key: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture
    (profiles/ncu_traffic.json, written by tools/ncu_summary.py from the .ncu-rep); None when no capture matches."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        e = t[kernel][key]
        return e["dram_read_bytes"] + e["dram_write_bytes"], e.get("source")
    except Exception:
        return None, None


def run_steps(sampler, latents, embeds, rope, n, step_i, inpaint=None):
    for _ in range(n):
        latents = sampler.step(latents, step_i, embeds, rope, inpaint)
        step_i += 1
    return latents, step_i


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--preset", default=os.environ.get("EA_BENCH_PRESET", "R720_7B"), choices=sorted(PRESETS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-vae", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the 12B / I2V / torch-baseline secondary lines")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the latents returned by the last timed step to DIR/latents.npy (float32), so that two builds "
                         "can be compared on the same seeded inputs")
    args = ap.parse_args()
    preset = PRESETS[args.preset]
    if args.impl == "reference":
        return run_reference_arm(args, preset)

    import torch
    from easyanimate_b200 import _lib, ops
    from easyanimate_b200.pipeline import EasyAnimateSampler, rope_table

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torchrun for N>1)"
    tiny = args.preset.startswith("tiny")
    assert args.warmup >= 3 or tiny, "timing rules: at least 3 warm-up steps"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    cfg_group = sp_group = world_group = None
    topology = os.environ.get("EA_BENCH_TOPOLOGY", "single_video")
    single_video = world >= 4 and topology != "replicas"
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        assert world % 2 == 0, "N>1 runs CFG-parallel pairs: N must be even"
        world_group = dist.group.WORLD
        if single_video:
            # ONE video on all N GPUs = 2 CFG branches x N/2 sequence-parallel ranks: ranks [0, P) evaluate the unconditional
            # branch, [P, 2P) the text branch; rank r and r + P form a CFG pair
            P = world // 2
            for b in range(2):  # every rank must create every group
                grp = dist.new_group(list(range(b * P, (b + 1) * P)))
                if rank // P == b:
                    sp_group = grp
            for r in range(P):
                grp = dist.new_group([r, r + P])
                if rank % P == r:
                    cfg_group = grp
        else:
            for g0 in range(0, world, 2):  # every rank must create every group
                grp = dist.new_group([g0, g0 + 1])
                if rank in (g0, g0 + 1):
                    cfg_group = grp

    def sync_all():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(*vals):
        t = torch.tensor(list(vals), device=dev, dtype=torch.float64)
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    bf16 = torch.bfloat16
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass

    def setup(preset_):
        """model + sampler + synthetic inputs of one preset under the run's topology"""
        F, h, w = preset_["F"], preset_["h"], preset_["w"]
        model = build_model(preset_, dev)
        if sp_group is not None:
            model.set_sequence_parallel_group(sp_group)
        sampler = EasyAnimateSampler(model, guidance_scale=GUIDANCE, cfg_group=cfg_group)
        rope = rope_table(h * 8, w * 8, F, device=dev)
        video_seed = 100 + (0 if (single_video or world == 1) else rank // 2)  # one video per CFG pair
        g = torch.Generator(device=dev).manual_seed(video_seed)
        latents = torch.randn((1, 16, F, h, w), device=dev, generator=g).to(bf16)
        embeds = (torch.randn((2, S_TEXT, E_TEXT), device=dev, generator=g) * 10).to(bf16)  # cat(negative, positive)
        inpaint = None
        if preset_.get("inpaint"):  # mask (1 channel) + masked-video latents (16), pipeline_easyanimate_inpaint.py:1496-1511
            inpaint = torch.randn((1, 17, F, h, w), device=dev, generator=g).to(bf16)
        return model, sampler, rope, latents, embeds, inpaint

    def timed_steps(sampler, latents, embeds, rope, inpaint, steps, warmup, collect_attn=False, clocks=None):
        sampler.set_timesteps(max(2 * (warmup + steps) + 8, 30), device="cpu")
        latents, i = run_steps(sampler, latents, embeds, rope, warmup, 0, inpaint)
        events = [] if collect_attn else None
        ops.ATTN_TIMING = events
        sync_all()
        if clocks is not None:
            clocks.start()  # sampled DURING the timed region only (warm-up and buffer set-up are over)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.ea_launch_count()
        e0.record()
        latents, i = run_steps(sampler, latents, embeds, rope, steps, i, inpaint)
        e1.record()
        sync_all()
        ops.ATTN_TIMING = None
        launches = _lib.ea_launch_count() - l0
        (ms,) = max_over_ranks(e0.elapsed_time(e1))
        attn_ms = [a.elapsed_time(b) for a, b in events] if events else []
        return ms, launches, attn_ms, latents, i

    # =============================================================================================================
    # headline: the preset's CFG step
    # =============================================================================================================
    F, h, w = preset["F"], preset["h"], preset["w"]
    model, sampler, rope, latents, embeds, inpaint = setup(preset)
    n_params = sum(p.numel() for p in model.parameters())
    clocks = ClockSampler(local_rank)
    ms_total, launches, attn_ms, latents, step_i = timed_steps(sampler, latents, embeds, rope, inpaint, args.steps, args.warmup, True,
                                                               clocks=clocks)
    clock_info = clocks.stop()
    if args.dump_outputs and rank == 0:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "latents.npy"), latents.float().cpu().numpy())

    # ---- end to end through the public API with HOST buffers (H2D inputs + D2H result every step)
    lat_host = torch.empty(latents.shape, dtype=bf16, pin_memory=True).copy_(latents)
    emb_host = torch.empty(embeds.shape, dtype=bf16, pin_memory=True).copy_(embeds)
    out_host = torch.empty(latents.shape, dtype=bf16, pin_memory=True)
    sampler.step_from_host(lat_host, step_i, emb_host, rope, out_host, device=dev, inpaint_latents=inpaint); step_i += 1  # warm
    sync_all()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(args.steps):
        sampler.step_from_host(lat_host, step_i, emb_host, rope, out_host, device=dev, inpaint_latents=inpaint); step_i += 1
        lat_host, out_host = out_host, lat_host
    f1.record()
    sync_all()
    (ms_e2e,) = max_over_ranks(f0.elapsed_time(f1))

    n_videos = 1 if (single_video or world == 1) else world // 2
    ms_per_step = ms_total / args.steps
    value = n_videos * args.steps / (ms_total / 1e3)
    e2e_value = n_videos * args.steps / (ms_e2e / 1e3)
    sp = world // 2 if single_video else 1

    line = None
    if rank == 0:
        peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
        peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"
        S = F * (h // 2) * (w // 2) + S_TEXT
        B_attn = 2 if cfg_group is None else 1
        heads_attn = preset["heads"] // sp  # Ulysses: heads sharded inside attention
        attn_flops = 4.0 * B_attn * heads_attn * S * S * 64
        attn_avg_ms = statistics.mean(attn_ms) if attn_ms else None
        achieved = attn_flops / (attn_avg_ms * 1e-3) / 1e12 if attn_avg_ms else None
        flops_step = 2 * dit_flops_per_forward(**_flop_args(preset))
        act_bytes = B_attn * S * preset["heads"] * 64 * 2  # one [B, S, d] bf16 activation
        traffic, traffic_src = load_traffic("attn6_kernel", f"B{B_attn}_H{heads_attn}_S{S}")
        if world == 1:
            par = "single GPU (CFG batch 2)"
        elif single_video:
            par = f"1 video on {world} GPUs: 2 CFG branches x {sp} sequence-parallel ranks (tokens sharded for per-token work, heads inside attention)"
        else:
            par = f"{n_videos} video(s) x CFG-parallel pair (1 all_gather of {latents.numel() * 2 / 1e6:.2f} MB per step)"
        line = {
            "metric": METRIC, "value": value, "unit": "steps/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak" if (world > 2 and not single_video) else "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": args.preset, "model": f"MMDiT d={preset['heads'] * 64} heads={preset['heads']} layers={preset['layers']}",
                       "params": n_params, "latent": [1, 16, F, h, w], "video": f"{4 * (F - 1) + 1}f {h * 8}x{w * 8}",
                       "tokens": S, "text_tokens": S_TEXT, "guidance_scale": GUIDANCE, "scheduler": "flow-match Euler shift=1",
                       "parallelism": par,
                       "l2": ("inputs_exceed_L2" if act_bytes > 126e6 else "inputs_fit_L2 (not a timing configuration)") +
                             f" (one activation tensor of a forward is {act_bytes / 1e6:.0f} MB, weights {n_params * 2 / 1e9:.1f} GB)",
                       "tflop_per_step": flops_step / 1e12,
                       "parity_criterion": "tests assert err(ours, fp32 truth) <= 1.5 x err(bf16 oracle, fp32 truth) + 2e-3 per module "
                                           "(a re-definition: north_star's rtol 1e-3 / atol 1e-4 is below one bf16 ulp and is only "
                                           "reported, tests/parity.py)"},
            "model_tflops": flops_step * value / 1e12, "forwards_per_s": 2.0 * value,  # a CFG step is two MMDiT forwards
            "e2e": {"value": e2e_value, "unit": "steps/s", "h2d_bytes_per_step": lat_host.numel() * 2 + emb_host.numel() * 2,
                    "d2h_bytes_per_step": out_host.numel() * 2},
            "gpu_launches": int(launches),
            "clocks": clock_info,
            "roofline": {"kernel": "a6::attn6_kernel (joint text+video attention, hd=64, ea_attn_args.variant 0x%x)" % ops.ATTN_VARIANT,
                         "bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": (achieved / peak_tf) if achieved else None, "peak_source": peak_src + " (of measured)",
                         "traffic": traffic, "traffic_source": traffic_src,
                         "traffic_algorithmic": 4.0 * B_attn * heads_attn * S * 64 * 2,
                         "launches_timed": len(attn_ms), "avg_ms": attn_avg_ms, "flops_per_launch": attn_flops,
                         "share_of_step": (sum(attn_ms) / ms_total) if attn_ms else None},
        }

    # ---- the whole call a user makes, end to end on ONE GPU: embeddings + noise from pinned host memory, K CFG steps,
    #      decode_latents, float32 frames in host memory (pipeline_easyanimate.py:1052-1149 after the text encoder)
    if rank == 0 and world == 1 and not args.no_vae:
        k_e2e = min(args.steps, 4)
        vae_e = build_vae(dev)
        sampler.vae = vae_e
        Tf = 4 * (F - 1) + 1
        frames = torch.empty((1, 3, Tf, 8 * h, 8 * w), dtype=torch.float32, pin_memory=True)

        def whole_call():
            lat = lat_host.to(dev, non_blocking=True)
            emb = emb_host.to(dev, non_blocking=True)
            sampler.set_timesteps(max(k_e2e, 1), device="cpu")
            for i in range(k_e2e):
                lat = sampler.step(lat, i, emb, rope, inpaint)
            return sampler.decode_latents(lat, out=frames)
        whole_call()  # warm
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        whole_call()
        g1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        ms_call = g0.elapsed_time(g1)
        line["e2e_video"] = {"steps": k_e2e, "ms": ms_call, "wall_s": wall, "frames_bytes_to_host": frames.numel() * 4,
                             "steps_per_s_including_decode": k_e2e / ms_call * 1e3, "finite": bool(torch.isfinite(frames).all()),
                             "what": f"{k_e2e} CFG steps + decode_latents (untiled) + float32 frames [1,3,{Tf},{8 * h},{8 * w}] in pinned "
                                     "host memory, inputs from pinned host memory; a 50-step call = 50 x ms_per_step + the decode tail"}
        sampler.vae = None
        del vae_e, frames
        torch.cuda.empty_cache()

    # =============================================================================================================
    # secondary lines (other BASELINE configs), all ranks take part when N > 1
    # =============================================================================================================
    secondary = {}
    model.set_sequence_parallel_group(None)  # (collective) unmaps the peers' exchange buffers before they are freed
    del model, sampler
    torch.cuda.empty_cache()
    want_secondary = not args.no_secondary and not tiny
    if want_secondary and args.preset != "R720_12B":
        # BASELINE configs[2]: 12B MMDiT at 49f 720x1280 (one video on all N GPUs)
        p12 = PRESETS["R720_12B"]
        m12, s12, rope12, lat12, emb12, _ = setup(p12)
        ms12, _, _, _, _ = timed_steps(s12, lat12, emb12, rope12, None, 3, 2)
        fl12 = 2 * dit_flops_per_forward(**_flop_args(p12))
        secondary["R720_12B"] = {"value": 3e3 / ms12 * (n_videos if not single_video else 1), "unit": "steps/s", "ms_per_step": ms12 / 3,
                                 "steps": 3, "warmup": 2, "params": sum(p.numel() for p in m12.parameters()),
                                 "model_tflops": fl12 * 3 / ms12 / 1e9 * (n_videos if not single_video else 1), "tflop_per_step": fl12 / 1e12}
        m12.set_sequence_parallel_group(None)
        del m12, s12
        torch.cuda.empty_cache()
    if want_secondary and world == 1:
        # BASELINE configs[4]: I2V 12B at 1024x1024x49: vae.encode of the conditioning video once, then the denoise step with
        # inpaint_latents (17 extra channels) - pipeline_easyanimate_inpaint.py:769-826,1320-1411,1522-1537
        pi = PRESETS["R1024_12B_I2V"]
        mi, si, ropei, lati, embi, inpi = setup(pi)
        msi, _, _, _, _ = timed_steps(si, lati, embi, ropei, inpi, 2, 2)
        fli = 2 * dit_flops_per_forward(**_flop_args(pi))
        secondary["R1024_12B_I2V"] = {"value": 2e3 / msi, "unit": "steps/s", "ms_per_step": msi / 2, "steps": 2, "warmup": 2,
                                      "tokens": pi["F"] * (pi["h"] // 2) * (pi["w"] // 2) + S_TEXT, "model_tflops": fli * 2 / msi / 1e9,
                                      "tflop_per_step": fli / 1e12}
        mi.set_sequence_parallel_group(None)
        del mi, si
        torch.cuda.empty_cache()

    if rank == 0 and world == 1 and not args.no_vae:
        vlines, vae = vae_lines(preset, dev, peaks)
        line["vae_decode"] = dict(vlines["untiled"], tiled=vlines["tiled"], e2e=vlines["e2e"])
        if want_secondary:
            # the I2V pipeline's one-off conditioning encode (configs[4]): 49 frames at 1024x1024
            try:
                x = (torch.rand((1, 3, 49, 1024, 1024), device=dev) * 2 - 1).to(bf16)
                ms_enc, post = time_cuda(lambda: vae.encode(x).latent_dist.mode(), 2)
                secondary["R1024_12B_I2V"]["vae_encode"] = {"ms": ms_enc, "MPix_per_s": 49 * 1024 * 1024 / 1e6 / ms_enc * 1e3,
                                                            "input": [1, 3, 49, 1024, 1024], "latent": list(post.shape)}
                del x, post
            except Exception as e:
                secondary["R1024_12B_I2V"]["vae_encode"] = {"unavailable": f"{type(e).__name__}: {str(e)[:160]}"}
        del vae
        torch.cuda.empty_cache()
    if world > 1 and not args.no_vae and not tiny:
        # tile-parallel tiled decode over ALL ranks (one all_gather of the decoded tiles), BASELINE configs[3] at N GPUs
        vae = build_vae(dev, tiled=True)
        vae.set_tile_parallel_group(world_group)
        z = (torch.randn((1, 16, F, h, w), device=dev, generator=torch.Generator(device=dev).manual_seed(5)) / 0.7125).to(bf16)
        vae.decode(z)
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        y = vae.decode(z).sample
        e1.record()
        sync_all()
        (ms_v,) = max_over_ranks(e0.elapsed_time(e1))
        if rank == 0:
            line["vae_decode"] = {"value": y.shape[2] * y.shape[3] * y.shape[4] / 1e6 / ms_v * 1e3, "unit": "MPix/s", "ms": ms_v,
                                  "mode": f"reference tiling, tiles sharded over {world} ranks, one all_gather, blend on every rank"}
        del y
        # the UNTILED decode of the same latent sharded by horizontal strips (easyanimate_b200/vae_strips.py: halo rows for the
        # convolutions, gathered GroupNorm sums, one all_gather of the frames): no 1.81x tiling overhead, the untiled result
        try:
            vae.use_tiling = False
            vae.set_tile_parallel_group(None)
            vae.set_strip_parallel_group(world_group)
            vae.decode(z)
            sync_all()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            y = vae.decode(z).sample
            e1.record()
            sync_all()
            (ms_s,) = max_over_ranks(e0.elapsed_time(e1))
            if rank == 0:
                line["vae_decode"]["strips"] = {"value": y.shape[2] * y.shape[3] * y.shape[4] / 1e6 / ms_s * 1e3, "unit": "MPix/s", "ms": ms_s,
                                                "finite": bool(torch.isfinite(y).all()),
                                                "mode": f"untiled decode, {world} horizontal strips (1 halo row per convolution and side, "
                                                        "GroupNorm sums all-gathered, one all_gather of the frames)"}
            del y
        except Exception as e:  # a secondary line must not take the headline down
            if rank == 0:
                line["vae_decode"]["strips"] = {"unavailable": f"{type(e).__name__}: {str(e)[:200]}"}
        del vae
        torch.cuda.empty_cache()

    if rank == 0:
        if want_secondary and world == 1:
            line["torch_gpu_baseline"] = torch_gpu_baseline(preset, dev)
        if secondary:
            line["secondary"] = secondary
        if world == 1 and not args.no_cpu_baseline:
            rate, desc, cores, _ = cpu_oracle_rate(seconds_budget=12.0)
            flops_step = 2 * dit_flops_per_forward(**_flop_args(preset))
            line["cpu_baseline"] = {"value": rate / flops_step, "unit": "steps/s", "cores": cores, "kind": "port", "sample": desc,
                                    "extrapolated": True}
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
