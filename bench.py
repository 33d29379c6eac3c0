#!/usr/bin/env python
"""bench.py -- motion-frames/sec of the full reverse-diffusion sampling loop (BASELINE.json metric).

One "step" = ONE pass of the hot path over one batch = one full sampling loop:
    body (pose) diffusion, 1000 steps (timestep_respacing ''), T = 600 frames, 104-dim pose,
    batch 8 per GPU (BASELINE configs[1]), CFG guidance 2.0 (sample/generate.py always wraps the
    model in ClassifierFreeSampleModel), random-init denoiser + synthetic wav2vec features.
value   = N*B*T / t_loop with inputs already resident in HBM (conditioning precompute is inside the loop time)
e2e     = same metric through the public API (Sampler.ddim_sample_loop) with HOST (pinned) inputs and a
          device->host read of the result inside the timed region
Scaling is weak: every rank owns B independent rows (no data-path collective; one all-gather of the result).

Besides the contract line (BASELINE configs[1]: B = 8 per GPU, weak scaling) every run also measures
  * "config3_strong": BASELINE configs[2] = the north-star's headline -- GLOBAL batch 32 + CFG, sharded over the N ranks
    (N = 1: batch 32 on one B200; N = 8: 4 rows per GPU = STRONG scaling of the same job),
  * "gpu_baseline" (rank 0, N = 1): the UNMODIFIED reference loop (oracle/_ref: ddim_sample_loop + ClassifierFreeSampleModel +
    FiLMTransformer, stock PyTorch fp32, TF32 off) on the same B200 -- the denominator of the north-star's ">= 10x" target,
  * "cpu_baseline": the same unmodified reference on the host cores (kind "reference"; the oracle port only if oracle/_ref
    is absent).

  python bench.py [--gpus N --steps K --warmup W]         this framework
  python bench.py --impl reference ...                      the reference's own loop on the host CPU cores (oracle/_ref)
  python bench.py --workload face ...                       BASELINE configs[3] (face, ddim500, g = 10, 16 rows / GPU): secondary
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from argparse import Namespace

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "motion-frames/sec full p_sample_loop (body, 1000 steps, T=600)"
UNIT = "frames/s"
WORKLOAD = dict(fmt="pose", layers=6, heads=8, T=600, S=1998, C=104, B=8, guidance=2.0, respacing="")
# BASELINE configs[3]: face diffusion, 500 steps (ddim500), T = 600, 256-dim codes, 16 rows per GPU (64 over 4 GPUs), g = 10
FACE_METRIC = "motion-frames/sec full ddim_sample_loop (face, ddim500, T=600)"
FACE_WORKLOAD = dict(fmt="face", layers=8, heads=8, T=600, S=1998, C=256, B=16, guidance=10.0, respacing="ddim500")
CONFIG3_GLOBAL_BATCH = 32


def workload_name(fmt, B, cfg, n_diff=None):
    if fmt == "pose":
        return (f"pose body diffusion, {n_diff or 1000} steps, T=600, C=104, batch {B}/GPU, {'CFG g=2.0' if cfg else 'NO CFG (bare denoiser)'}, "
                f"L=6 D=256 H=8, synthetic wav2vec features [B,1998,1024] (BASELINE configs[1])")
    return (f"face diffusion, {n_diff or 500} steps (ddim500), T=600, C=256, batch {B}/GPU, CFG g=10.0, L=8 D=512 H=8, synthetic "
            f"audio+lip features [B,1998,2038] (BASELINE configs[3])")


SPLIT_TERMS = 2


def model_args(respacing):
    return Namespace(split_terms=SPLIT_TERMS, data_format="pose", add_frame_cond=1, max_seq_length=600, layers=WORKLOAD["layers"],
                     heads=WORKLOAD["heads"], not_rotary=False, unconstrained=False, device="cuda",
                     timestep_respacing=respacing, noise_schedule="cosine", sigma_small=True, lambda_vel=0.0,
                     model_path="synthetic", resume_trans=None)


def synth_inputs(B, T, S, seed, pin=False):
    g = torch.Generator().manual_seed(seed)
    y = {
        "audio_embed": torch.randn(B, S, 1024 if WORKLOAD["fmt"] == "pose" else 2038, generator=g),
        "keyframes": torch.randn(B, len(range(0, T, 30)), 104, generator=g),
        "mask": torch.ones(B, 1, 1, T, dtype=torch.bool),
        "scale": torch.full((B,), WORKLOAD["guidance"]),
    }
    noise = torch.randn(B, WORKLOAD["C"], 1, T, generator=g)
    if pin and torch.cuda.is_available():
        y = {k: v.pin_memory() for k, v in y.items()}
        noise = noise.pin_memory()
    return y, noise


def flops_per_sample_forward(T=600, S=2000, S2=20, D=256, L=6, FF=1024, C=104, fmt="pose"):
    """SURVEY.md 8d formulas (2*MAC, cached-K/V convention); face: no keyframe attention, no TCN, 3 FiLM blocks."""
    sa = 6 * T * D * D + 4 * T * T * D + 2 * T * D * D
    ca = 2 * T * D * D + 8 * D * D + 4 * T * S * D + 2 * T * D * D
    ffn = 4 * T * D * FF
    io = 4 * T * C * D
    if fmt == "face":
        return L * (sa + ca + ffn + 3 * 4 * D * D) + io + 32 * D * D
    ca2 = 2 * T * D * D + 4 * T * S2 * D + 2 * T * D * D
    film = 4 * 4 * D * D
    lens = [T + 24 - 2, T + 24 - 6, T + 24 - 12, T + 24 - 14, T + 24 - 18, T]
    ch = [(104, 256), (256, 104), (104, 104), (104, 104), (104, 104), (104, 104)]
    conv = sum(2 * ln * ci * co * 3 for ln, (ci, co) in zip(lens, ch)) + 2 * T * C * C
    return L * (sa + ca + ca2 + ffn + film) + io + conv + 32 * D * D


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.proc.wait()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[2:6]) if v.lower() == "active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


CPU_SAMPLE_STEPS = 10  # diffusion steps the oracle-PORT fallback times
CPU_SAMPLE_ROWS = 2


def cpu_port_frames_per_s(n_diff_steps, threads):
    """FALLBACK (oracle/_ref absent): the reference's algorithm as restated by the oracle, on a bounded sample
    (`n_diff_steps` CFG steps of CPU_SAMPLE_ROWS of the 8 rows, scaled to 8 rows x 1000 steps)."""
    from oracle import a2p_oracle as O
    from audio2photoreal_b200.weights import model_dims, synthetic_state_dict
    torch.set_num_threads(threads)
    w = WORKLOAD
    sd = synthetic_state_dict(model_dims("pose", w["layers"], w["heads"]), seed=1)
    y, noise = synth_inputs(CPU_SAMPLE_ROWS, w["T"], w["S"], seed=10)
    od = O.OracleDiffusion("")
    fn = lambda x, ts: O.cfg_forward(sd, "pose", w["heads"], x, ts, y["audio_embed"], y["keyframes"], y["mask"], y["scale"])
    with torch.no_grad():
        od.ddim_sample_loop(fn, noise, skip_timesteps=999)       # warm-up: one step
        t0 = time.perf_counter()
        od.ddim_sample_loop(fn, noise, skip_timesteps=1000 - n_diff_steps)
        dt = time.perf_counter() - t0
    per_step_full_batch = dt / n_diff_steps * (w["B"] / CPU_SAMPLE_ROWS)
    return w["B"] * w["T"] / (per_step_full_batch * 1000), dt


class ReferenceLoop:
    """The UNMODIFIED reference on this box: oracle/_ref (byte-for-byte view written by oracle/build_ref.py) imported
    through oracle/ref_harness.py's shims (stand-in fairseq conv stack of the published geometry, scratch cwd).  One call =
    `k` diffusion steps of the reference's own `ddim_sample_loop` (skip_timesteps = N - k: the last k indices of the
    1000-step schedule; per-step cost is shape-static) with ClassifierFreeSampleModel and RAW 48 kHz audio, i.e. including
    the per-call `encode_audio` the reference pays twice per step (model/diffusion.py:355-358)."""

    def __init__(self, device: str, batch: int, fmt: str = "pose"):
        import contextlib
        with contextlib.redirect_stdout(sys.stderr):      # the reference prints while it builds; stdout carries ONE JSON line
            self._init(device, batch, fmt)

    def _init(self, device: str, batch: int, fmt: str):
        from oracle import ref_harness as RH
        from audio2photoreal_b200.weights import model_dims, synthetic_state_dict
        w = WORKLOAD if fmt == "pose" else FACE_WORKLOAD
        self.w, self.B, self.dev = w, batch, torch.device(device)
        sd = synthetic_state_dict(model_dims(fmt, w["layers"], w["heads"]), seed=1)
        self.ref, self.args, model, self.diffusion = RH.build_reference(fmt, w["layers"], w["heads"], w["respacing"], sd, device=device)
        self.model = self.ref.cfg.ClassifierFreeSampleModel(model).to(self.dev).eval()
        g = torch.Generator().manual_seed(10)
        T = w["T"]
        self.y = {"audio": (0.1 * torch.randn(batch, T * 1600, 2, generator=g)).to(self.dev),
                  "keyframes": torch.randn(batch, len(range(0, T, 30)), 104, generator=g).to(self.dev),
                  "mask": torch.ones(batch, 1, 1, T, dtype=torch.bool, device=self.dev),
                  "scale": torch.full((batch,), w["guidance"], device=self.dev)}
        self.noise = torch.randn(batch, w["C"], 1, T, generator=g).to(self.dev)
        self.n = self.diffusion.num_timesteps
        if self.dev.type == "cuda":
            torch.backends.cuda.matmul.allow_tf32 = False      # the reference never enables TF32 (SURVEY 2a)
            torch.backends.cudnn.allow_tf32 = False
        else:
            import contextlib
            self._cuda_shim = True

    def run(self, k: int) -> float:
        """seconds for k diffusion steps (wall clock; device-synchronised on CUDA)"""
        import contextlib
        shim = contextlib.nullcontext()
        if self.dev.type != "cuda":       # model/diffusion.py:321 hard-codes .cuda(): neutralised for the CPU arm only
            old = torch.Tensor.cuda

            @contextlib.contextmanager
            def _s():
                torch.Tensor.cuda = lambda t, *a, **kk: t
                try:
                    yield
                finally:
                    torch.Tensor.cuda = old
            shim = _s()
        if self.dev.type == "cuda":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        with torch.no_grad(), shim, contextlib.redirect_stdout(sys.stderr):
            out = self.diffusion.ddim_sample_loop(self.model, (self.B, self.w["C"], 1, self.w["T"]), noise=self.noise,
                                                  clip_denoised=False, model_kwargs={"y": dict(self.y)},
                                                  skip_timesteps=self.n - k, init_image=None, progress=False)
        if self.dev.type == "cuda":
            torch.cuda.synchronize()
        assert torch.isfinite(out).all()
        return time.perf_counter() - t0

    def frames_per_s(self, k: int, reps: int = 1):
        ts = [self.run(k) for _ in range(reps)]
        t = float(np.median(ts))
        return self.B * self.w["T"] / (t / k * self.n), t


def reference_view_available() -> bool:
    try:
        from oracle import ref_harness as RH
        return RH.reference_available()
    except Exception:
        return False


def host_threads() -> int:
    return min(os.cpu_count() or 1, 32)    # torch CPU GEMMs of this size stop scaling (and regress) beyond ~32 threads


def cpu_baseline(fmt: str = "pose"):
    """cpu_baseline object of the bench line: bounded sample (1 warm-up + 2 timed diffusion steps of all 8 rows, ~10-30 s)."""
    threads = host_threads()
    torch.set_num_threads(threads)
    w = WORKLOAD if fmt == "pose" else FACE_WORKLOAD
    if reference_view_available():
        rl = ReferenceLoop("cpu", w["B"], fmt)
        rl.run(1)
        v, t = rl.frames_per_s(2)
        return {"value": v, "unit": UNIT, "cores": threads, "kind": "reference",
                "sample": f"2 of {rl.n} diffusion steps (after 1 warm-up step) of all {w['B']} rows through the reference's own "
                          f"ddim_sample_loop + ClassifierFreeSampleModel + FiLMTransformer (oracle/_ref; raw 48 kHz audio, stand-in "
                          f"wav2vec conv stack, encode_audio paid per call like the reference) in {t:.1f}s, scaled x{rl.n}/2"}
    v, dt = cpu_port_frames_per_s(CPU_SAMPLE_STEPS, threads)
    return {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{CPU_SAMPLE_STEPS} of 1000 diffusion steps of {CPU_SAMPLE_ROWS} of the 8 batch rows (oracle port, synthetic features) "
                      f"in {dt:.1f}s, scaled x1000/{CPU_SAMPLE_STEPS} x 8/{CPU_SAMPLE_ROWS}"}


def gpu_baseline(batch: int, k: int = 10):
    """The reference GPU path (BASELINE.md 3.4): unmodified reference loop on this B200, stock PyTorch fp32."""
    if not reference_view_available():
        return None
    try:
        rl = ReferenceLoop("cuda", batch)
        rl.run(2)
        v, t = rl.frames_per_s(k, reps=3)
        del rl
        torch.cuda.empty_cache()
        return {"value": v, "unit": UNIT, "kind": "reference", "batch": batch,
                "sample": f"median of 3 x {k} of 1000 diffusion steps (after 2 warm-up steps) of the reference's own loop on cuda, fp32, "
                          f"TF32 off, batch {batch} + CFG, raw-audio encode per call, {t:.2f}s per {k} steps, scaled x1000/{k}"}
    except Exception as e:       # never let the baseline leg take the bench line down
        return {"value": None, "unit": UNIT, "kind": "reference", "batch": batch, "error": repr(e)[:200]}


def run_reference_arm(a):
    """--impl reference: every bench "step" is a bounded sample (ONE diffusion step of all 8 rows through the reference's own
    public API on the host cores); value = B*T / (median step time x 1000 steps)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    torch.set_num_threads(threads)
    fmt = "face" if a.workload == "face" else "pose"
    w = WORKLOAD if fmt == "pose" else FACE_WORKLOAD
    if reference_view_available():
        rl = ReferenceLoop("cpu", w["B"], fmt)
        for _ in range(max(1, min(a.warmup, 2))):
            rl.run(1)
        ts = [rl.run(1) for _ in range(max(1, a.steps))]
        t = float(np.median(ts))
        v = w["B"] * w["T"] / (t * rl.n)
        kind = "reference"
        sample = (f"each of the {a.steps} timed steps = 1 of {rl.n} diffusion steps of all {w['B']} rows through the reference's own "
                  f"ddim_sample_loop (oracle/_ref, raw audio, encode_audio per call), median {t:.2f}s, scaled x{rl.n}")
    else:
        vals = [cpu_port_frames_per_s(5, threads)[0] for _ in range(max(1, a.steps))]
        v, kind = float(np.median(vals)), "port"
        sample = "oracle port: 5 of 1000 steps of 2 of 8 rows, scaled (oracle/_ref absent)"
    line = {
        "impl": "reference", "metric": METRIC if fmt == "pose" else FACE_METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * w["B"] * w["T"] / v, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(fmt, w["B"], True).replace("synthetic wav2vec features [B,1998,1024]", "synthetic RAW 48 kHz audio "
                                                                       "[B,960000,2] through the stand-in vq-wav2vec stack on every call")},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir, **arrays):
    """<out_dir>/<name>.npy in float32, one file per output array"""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


# ---------------------------------------------------------------- BASELINE configs[4]: the full pipeline of one subject per GPU
PIPE_METRIC = "motion-frames/sec full pipeline (guide keyframes + body 1000 steps + face ddim500, T=600)"
PIPE_SAMPLES = 16          # samples per subject (configs[4]: 4 subjects x 16 samples)


def _synthetic_guide(dev, tokens=1024, dim=512, layers=4, depth=4, latent=64):
    """GuideSampler + VQDecoder with random weights under the reference's checkpoint key names (model/guide.py, model/vqvae.py) and
    a random-init frozen extractor of the published vq-wav2vec conv geometry (there are no checkpoints offline)."""
    import torch.nn as nn
    from audio2photoreal_b200.guide import GuideSampler, VQDecoder
    g = torch.Generator().manual_seed(5)
    rn = lambda *sh, sc=1.0: torch.randn(*sh, generator=g) * sc

    class Extractor(nn.Module):
        def __init__(self):
            super().__init__()
            geo, cin, mods = [(512, 10, 5), (512, 8, 4), (512, 4, 2), (512, 4, 2), (512, 4, 2), (512, 1, 1), (512, 1, 1), (512, 1, 1)], 1, []
            for d_, k, st in geo:
                mods.append(nn.Sequential(nn.Conv1d(cin, d_, k, stride=st, bias=False), nn.GroupNorm(1, d_), nn.ReLU()))
                cin = d_
            self.conv_layers = nn.ModuleList(mods)

        def feature_extractor(self, x):
            x = x.unsqueeze(1)
            for c in self.conv_layers:
                x = c(x)
            return torch.log(torch.abs(x) + 1)
    sd = {"token_embedding.weight": rn(tokens + 1, dim), "rotary.freqs": 1.0 / (10000 ** (torch.arange(0, dim, 2).float() / dim)),
          "audio_resampler.kernel": rn(1, 1, 41, sc=1 / 41), "null_cond_embed": rn(1, 798, dim), "null_cond_hidden": rn(1, dim),
          "norm_cond.weight": torch.ones(dim), "norm_cond.bias": torch.zeros(dim),
          "cond_projection.weight": rn(dim, 1024, sc=1024 ** -0.5), "cond_projection.bias": torch.zeros(dim),
          "non_attn_cond_projection.0.weight": torch.ones(dim), "non_attn_cond_projection.0.bias": torch.zeros(dim),
          "non_attn_cond_projection.1.weight": rn(dim, dim, sc=dim ** -0.5), "non_attn_cond_projection.1.bias": torch.zeros(dim),
          "non_attn_cond_projection.3.weight": rn(dim, dim, sc=dim ** -0.5), "non_attn_cond_projection.3.bias": torch.zeros(dim),
          "final_layer.weight": rn(tokens, dim, sc=dim ** -0.5), "final_layer.bias": torch.zeros(tokens)}
    idx = 0
    for _ in range(2):                      # num_audio_layers = 2 blocks of six dilated convs (model/guide.py:84-119)
        for _ in range(6):
            sd[f"pre_audio.{idx}.weight"], sd[f"pre_audio.{idx}.bias"] = rn(1024, 1024, 3, sc=(3 * 1024) ** -0.5), torch.zeros(1024)
            idx += 3
    sd[f"pre_audio.{idx}.weight"], sd[f"pre_audio.{idx}.bias"] = rn(1024, 1024, 1, sc=1024 ** -0.5), torch.zeros(1024)
    for n in range(layers):
        p_ = f"seqTransDecoder.stack.{n}."
        for a_ in ("self_attn", "multihead_attn"):
            sd[p_ + a_ + ".in_proj_weight"], sd[p_ + a_ + ".in_proj_bias"] = rn(3 * dim, dim, sc=dim ** -0.5), torch.zeros(3 * dim)
            sd[p_ + a_ + ".out_proj.weight"], sd[p_ + a_ + ".out_proj.bias"] = rn(dim, dim, sc=dim ** -0.5), torch.zeros(dim)
        sd[p_ + "linear1.weight"], sd[p_ + "linear1.bias"] = rn(1024, dim, sc=dim ** -0.5), torch.zeros(1024)
        sd[p_ + "linear2.weight"], sd[p_ + "linear2.bias"] = rn(dim, 1024, sc=1024 ** -0.5), torch.zeros(dim)
        for k in ("norm1", "norm2", "norm3"):
            sd[p_ + k + ".weight"], sd[p_ + k + ".bias"] = torch.ones(dim), torch.zeros(dim)
        for k in ("film1", "film2", "film3"):
            sd[p_ + k + ".block.1.weight"], sd[p_ + k + ".block.1.bias"] = rn(2 * dim, dim, sc=dim ** -0.5), torch.zeros(2 * dim)
        sd[p_ + "rotary.freqs"] = sd["rotary.freqs"].clone()
    guide = GuideSampler(sd, tokens=tokens, audio_model=Extractor()).to(dev).eval()
    vq = {f"quantizer.layers.{i}._codebook.embed": rn(tokens, latent) for i in range(depth)}
    for i in (0, 2, 4, 6):
        vq[f"decoder.dec.{i}.weight"], vq[f"decoder.dec.{i}.bias"] = rn(latent, latent, 2, sc=(2 * latent) ** -0.5), torch.zeros(latent)
    vq["decoder.dec.8.weight"], vq["decoder.dec.8.bias"] = rn(104, latent, 1, sc=latent ** -0.5), torch.zeros(104)
    return guide, VQDecoder(vq, 104, latent, tokens, depth).to(dev).eval()


def run_pipeline(a):
    """One subject per GPU (4 subjects on 4 GPUs; 8 GPUs = the 4 subjects' face and body jobs would be the alternative cut):
    guide keyframes (KV-cached AR sampler + VQ decode, sample/generate.py:51-71) -> body diffusion (1000 steps, g = 2) with those
    keyframes -> face diffusion (ddim500, g = 10), 16 samples per subject, T = 600; value = N x 16 x 600 frames / time."""
    import torch.distributed as dist
    from audio2photoreal_b200.api import CFGDenoiser, create_model_and_diffusion, load_model
    from audio2photoreal_b200.dist import all_gather_rows
    from audio2photoreal_b200.weights import synthetic_state_dict
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, T = PIPE_SAMPLES, 600
    guide, vq = _synthetic_guide(dev)
    models = {}
    for fmt, resp, g_ in (("pose", "", 2.0), ("face", "ddim500", 10.0)):
        m = model_args(resp)
        m.split_terms = 2 if fmt == "pose" else 3
        if fmt == "face":
            m.data_format, m.add_frame_cond = "face", None
            m.layers = FACE_WORKLOAD["layers"]
        model, sampler = create_model_and_diffusion(m, "test")
        load_model(model, synthetic_state_dict(model.dims, seed=1))
        model = model.to(dev).eval()
        models[fmt] = (model, CFGDenoiser(model), sampler, g_)
    gen = torch.Generator().manual_seed(20 + rank)
    audio = (0.1 * torch.randn(B, T * 1600, 2, generator=gen)).pin_memory()
    feats = {"pose": torch.randn(B, 1998, 1024, generator=gen).pin_memory(), "face": torch.randn(B, 1998, 2038, generator=gen).pin_memory()}
    noise = {"pose": torch.randn(B, 104, 1, T, generator=gen).pin_memory(), "face": torch.randn(B, 256, 1, T, generator=gen).pin_memory()}

    def once():
        a_dev = audio.to(dev, non_blocking=True)
        toks = guide.generate(a_dev, T // 30, layers=vq.residual_depth, n_sequences=B)            # sample/generate.py:60-66
        keyframes = vq.decode(toks.reshape(B, -1, vq.residual_depth))                              # :67-70 -> [B, 20, 104]
        out = {}
        for fmt in ("pose", "face"):
            model, cfg, sampler, g_ = models[fmt]
            y = {"audio_embed": feats[fmt].to(dev, non_blocking=True), "keyframes": keyframes.clone(), "mask": torch.ones(B, 1, 1, T, dtype=torch.bool),
                 "scale": torch.full((B,), g_, device=dev)}
            model._cond_sig = None
            out[fmt] = sampler.ddim_sample_loop(cfg, (B, model.nfeats, 1, T), noise=noise[fmt].to(dev, non_blocking=True), clip_denoised=False,
                                                model_kwargs={"y": y}, advance_rng=False)
        res = torch.cat([out["pose"], out["face"]], dim=1)                                       # [B, 104 + 256, 1, T]
        return all_gather_rows(res, B * world).cpu()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(max(1, min(a.warmup, 2))):
        once()
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        res = once()
    torch.cuda.synchronize()
    dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    barrier()
    assert torch.isfinite(res).all() and res.shape[0] == B * world
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, sample=res)
    if rank == 0:
        ms = dt.item() * 1e3 / a.steps
        v = world * B * T / (ms / 1e3)
        line = {"metric": PIPE_METRIC, "value": v, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16x2 (pose) / bf16x3 (face) split, fp32 accumulate",
                "data": "synthetic",
                "config": {"workload": f"full pipeline per subject and GPU: guide AR sampler (80 tokens, KV cache) + VQ decode -> body diffusion 1000 steps g=2 -> "
                                       f"face diffusion ddim500 g=10; {B} samples x T=600 per subject, {world} subject(s) (BASELINE configs[4]); random-init weights, "
                                       f"raw audio for the guide, synthetic wav2vec(+lip) features for the denoisers",
                           "global_batch": B * world, "parallelism": f"one subject per GPU x{world}, 1 all-gather"},
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": int(audio.numel() * 4 + sum(t.numel() * 4 for t in feats.values()) + sum(t.numel() * 4 for t in noise.values())),
                        "d2h_bytes_per_step": int(res.numel() * 4 // world)},
                "gpu_launches": int(sum(m[0].launch_count() for m in models.values())), "roofline": None, "cpu_baseline": None}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    global SPLIT_TERMS, WORKLOAD, METRIC
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="a2p", choices=["a2p", "reference"])
    ap.add_argument("--diffusion-steps", type=int, default=1000, help="debug only; anything but 1000 is not the benchmark")
    ap.add_argument("--batch", type=int, default=WORKLOAD["B"], help="debug only; per-GPU batch")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cfg", action="store_true",
                    help="secondary measurement (SURVEY 8d, config 2 'no-CFG variant'): the bare denoiser, one forward per step; "
                         "not the benchmark line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned to its caller as DIR/<name>.npy (float32), so that two builds "
                         "can be compared output for output: the inputs depend only on the arguments")
    ap.add_argument("--split-terms", type=int, default=None, help="0: exact-fp32 FFMA arm; 2 (pose default, fused chain kernels) | 3 (face default): split-bf16 tcgen05 arms")
    ap.add_argument("--workload", default="pose", choices=["pose", "face", "pipeline"],
                    help="pose = BASELINE configs[1] (the contract line); face = configs[3] (ddim500, g=10, 16 rows/GPU); pipeline = configs[4] "
                         "(guide + body + face per subject and GPU); the last two are secondary")
    ap.add_argument("--no-config3", action="store_true", help="skip the extra global-batch-32 (configs[2], strong-scaling) measurement")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip the reference-on-this-GPU leg")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs: the reference arm times single diffusion steps, not whole loops")
    face = a.workload == "face"
    SPLIT_TERMS = a.split_terms if a.split_terms is not None else (3 if face else 2)
    if a.impl == "reference":
        return run_reference_arm(a)
    if a.workload == "pipeline":
        return run_pipeline(a)
    if face:
        if a.batch == WORKLOAD["B"]:
            a.batch = FACE_WORKLOAD["B"]
        if a.diffusion_steps == 1000:
            a.diffusion_steps = 500
        WORKLOAD, METRIC = FACE_WORKLOAD, FACE_METRIC
        a.no_config3 = True

    import torch.distributed as dist
    from audio2photoreal_b200 import _lib
    from audio2photoreal_b200.api import CFGDenoiser, create_model_and_diffusion, load_model
    from audio2photoreal_b200.dist import all_gather_rows
    from audio2photoreal_b200.weights import synthetic_state_dict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    w = WORKLOAD
    B, T, S = a.batch, w["T"], w["S"]
    resp = "" if a.diffusion_steps == 1000 else f"ddim{a.diffusion_steps}"
    margs = model_args(resp)
    if face:
        margs.data_format, margs.add_frame_cond = "face", None
    model, sampler = create_model_and_diffusion(margs, "test")
    load_model(model, synthetic_state_dict(model.dims, seed=1))
    model = model.to(dev).eval()
    cfg = model if a.no_cfg else CFGDenoiser(model)
    nbr = 1 if a.no_cfg else 2          # denoiser evaluations per row and step
    n_diff = sampler.num_timesteps
    shape = (B, w["C"], 1, T)

    # per-rank inputs (rank-dependent seed: independent rows on every GPU = weak scaling)
    def make_loops(Bl, n_rows_global, seed):
        y_host, noise_host = synth_inputs(Bl, T, S, seed=seed, pin=True)
        y_dev = {k: v.to(dev) for k, v in y_host.items()}
        noise_dev = noise_host.to(dev)
        shp = (Bl, w["C"], 1, T)

        def loop_resident():
            yy = dict(y_dev)
            model._cond_sig = None          # drop the conditioning cache: the one-time precompute is part of every loop
            res = sampler.ddim_sample_loop(cfg, shp, noise=noise_dev, clip_denoised=False, model_kwargs={"y": yy},
                                           advance_rng=False)
            return all_gather_rows(res, n_rows_global)     # the one collective of the path (no-op at world size 1)

        def loop_e2e():
            yy = {k: v.to(dev, non_blocking=True) for k, v in y_host.items()}
            nz = noise_host.to(dev, non_blocking=True)
            model._cond_sig = None
            res = sampler.ddim_sample_loop(cfg, shp, noise=nz, clip_denoised=False, model_kwargs={"y": yy}, advance_rng=False)
            return all_gather_rows(res, n_rows_global).cpu()
        loop_e2e.is_e2e = True
        h2d = sum(v.numel() * v.element_size() for v in y_host.values()) + noise_host.numel() * 4
        return loop_resident, loop_e2e, h2d, y_dev

    loop_resident, loop_e2e, h2d, y_dev = make_loops(B, B * world, 10 + rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(k):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        ms = max(e0.elapsed_time(e1), 0.0)
        ms = max(ms, wall * 1e3) if getattr(fn, "is_e2e", False) else ms    # e2e includes the host-side result copy
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        barrier()
        return t.item() / k, out

    for _ in range(a.warmup):
        loop_resident()
    launches0 = model.launch_count()
    clocks = ClockSampler(local)
    clocks.start()
    try:
        ms_step, out = timed(loop_resident, a.steps)
    finally:
        clk = clocks.stop()
    launches = (model.launch_count() - launches0)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, sample=out)
    loop_e2e()
    ms_e2e, out_h = timed(loop_e2e, a.steps)
    assert out.shape[0] == B * world and torch.isfinite(out).all()

    frames = world * B * T
    value = frames / (ms_step / 1e3)
    e2e_value = frames / (ms_e2e / 1e3)
    d2h = out_h.numel() * 4

    # ---- BASELINE configs[2] (north-star headline): GLOBAL batch 32 + CFG sharded over the N ranks = strong scaling of one job
    config3 = None
    if not a.no_config3 and not a.no_cfg:
        from audio2photoreal_b200.dist import shard_range
        lo, hi = shard_range(CONFIG3_GLOBAL_BATCH, world, rank)
        l3, l3e, h2d3, y_dev3 = make_loops(hi - lo, CONFIG3_GLOBAL_BATCH, 100 + rank)
        l3()
        k3 = max(2, min(a.steps, 5))
        ms3, out3 = timed(l3, k3)
        ms3e, out3h = timed(l3e, 2)
        assert out3.shape[0] == CONFIG3_GLOBAL_BATCH and torch.isfinite(out3).all()
        f3 = CONFIG3_GLOBAL_BATCH * T
        config3 = {"workload": f"pose body diffusion + CFG g=2.0, {n_diff} steps, T=600, GLOBAL batch {CONFIG3_GLOBAL_BATCH} sharded over {world} GPU(s) "
                               f"({hi - lo} rows on rank 0), audio K/V cached across steps (BASELINE configs[2])",
                   "scaling": "strong", "global_batch": CONFIG3_GLOBAL_BATCH, "n_gpus": world, "steps": k3,
                   "value": f3 / (ms3 / 1e3), "unit": UNIT, "ms_per_step": ms3,
                   "e2e": {"value": f3 / (ms3e / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(h2d3), "d2h_bytes_per_step": int(out3h.numel() * 4)}}
        del l3, l3e, out3, out3h

    roofline, cpu_base = None, None
    if rank == 0:
        # ---- live per-kernel measurement (CUDA events around every launch of one denoiser evaluation)
        lib = _lib.load()
        model._cond_sig = None
        model.prepare(dict(y_dev), B, T, dev)      # conditioning of the contract workload (config3 above changed it)
        # one-time cost per distinct y (inside every timed loop above): native conditioning encoders + K/V-cache build
        ce0, ce1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ce0.record()
        for _ in range(3):
            model._cond_sig = None
            model.prepare(dict(y_dev), B, T, dev)
        ce1.record()
        torch.cuda.synchronize()
        cond_ms = ce0.elapsed_time(ce1) / 3
        ncat = 9
        ms_cat = (C.c_float * ncat)()
        n_cat = (C.c_int64 * ncat)()
        n_cat_c = n_cat                      # the ctypes array (n_cat is rebound to a list of ints below)
        x_btc = torch.randn(B, T, w["C"], device=dev)
        ts = torch.full((B,), 500, device=dev, dtype=torch.int64)
        ws = model._workspace(lib.a2p_workspace_bytes(C.byref(model._cfg), B, T), dev)
        acc = np.zeros(ncat)
        reps = 5
        # the fused arm cuts a CFG step into concurrent forwards: {cond, uncond} x groups of batch rows (engine.cu,
        # sample_loop_impl).  Profile the launches the loop really makes -- every (branch, row group) forward, every launch
        # timed ALONE (in the loop the units overlap, so the per-kernel times add up to more than a step)
        groups = int(lib.a2p_loop_row_groups(model._handle, B, T))      # 0: one stacked forward for both branches
        units = [(3, 0, B)] if groups == 0 else [(mk, B * g // groups, B * (g + 1) // groups - B * g // groups)
                                                 for g in range(groups) for mk in (1, 2)]
        if a.no_cfg:
            groups, units = 0, [(1, 0, B)]
        two_branch = groups > 0
        rows_per_launch = nbr * B if groups == 0 else units[0][2]
        n_tot = np.zeros(ncat, dtype=np.int64)
        for i in range(reps + 1):
            for mk, b0, bs in units:
                _lib.check(lib.a2p_profile_forward_rows(model._handle, B, b0, bs, T, x_btc[b0:].data_ptr(), ts[b0:].data_ptr(), mk,
                                                        ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream,
                                                        ms_cat, n_cat, ncat))
                if i:
                    acc += np.array(list(ms_cat))
                if i == 1:
                    n_tot += np.array(list(n_cat), dtype=np.int64)
        acc /= reps
        n_cat = [int(v) for v in n_tot]
        names = ["cond_gemm", "ln_rope", "attn_proj_gemm", "attn_self", "attn_cross_audio", "attn_cross_keyframe", "ffn_gemm",
                 "io_tcn_gemm", "misc"]
        # kernel families: the three attention categories are launches of ONE kernel (umma_attn2_kernel), likewise the
        # chain categories; the dominant kernel is the family with the largest share of the step, reported through its
        # biggest category (the audio cross-attention launch / the FFN chain launches)
        fam_attn, fam_chain = acc[3] + acc[4] + acc[5], acc[2] + acc[6]
        dom = (4 if fam_attn >= fam_chain else int(np.argmax([0, 0, acc[2], 0, 0, 0, acc[6]]))) if SPLIT_TERMS == 2 else int(np.argmax(acc))
        R = nbr * B        # rows of one step (both branches); per-launch figures below divide by the launch counts
        D, L = model.dims.D, w["layers"]
        # per-launch algorithmic FLOPs of each category (attention cores exactly; linears = category total / launches)
        lin_proj = (16 if w["fmt"] == "pose" else 12) * T * D * D * R * L
        lin_ffn = 4 * T * D * 1024 * R * L
        if SPLIT_TERMS == 2:   # fused chain arm: PROJ = {sa_out+q, ca_out+q} per layer, FFN = {out+ffn1, ffn2+next qkv} per layer
            lin_proj, lin_ffn = 8 * T * D * D * R * L, (2 * T * D * D + 4 * T * D * 1024 + 6 * T * D * D) * R * L
        alg = {3: 4 * T * T * D * R * L / max(1, n_cat[3]), 4: 4 * T * (S + 2) * D * R * L / max(1, n_cat[4]),
               5: 4 * T * 20 * D * R * L / max(1, n_cat[5]),
               2: lin_proj / max(1, n_cat[2]), 6: lin_ffn / max(1, n_cat[6])}
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_tf = peaks.get("bf16_tflops", 1590.0)
        peak_src = "measured" if "bf16_tflops" in peaks else "fallback"
        per_launch_ms = acc[dom] / max(1, n_cat[dom])
        flops_launch = alg.get(dom, 0)
        achieved = flops_launch / (per_launch_ms * 1e-3) / 1e12 if per_launch_ms > 0 else 0.0
        traffic = None     # DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")))
            if tr.get("kernel") == names[dom] and B == WORKLOAD["B"] and tr.get("rows_per_launch", 2 * B) == rows_per_launch:
                traffic = tr["dram_bytes_per_launch"]
        except Exception:
            pass
        roofline = {"bound": "tensor", "kernel": names[dom], "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": achieved / peak_tf, "traffic": traffic, "peak_source": f"bf16_tflops burst, of {peak_src}",
                    "ms_per_launch": per_launch_ms, "launches_per_forward": int(n_cat[dom]),
                    "forward_ms_by_kernel": {n: round(float(v), 4) for n, v in zip(names, acc)},
                    "kernel_family_ms": {"attention(self+audio+keyframe)": round(float(fam_attn), 4), "chain(proj+ffn)": round(float(fam_chain), 4)},
                    "split_terms": SPLIT_TERMS,
                    "launch_shape": ("bare denoiser, no CFG: one forward of B rows per step" if a.no_cfg else f"{rows_per_launch} rows of one CFG branch per launch ({len(units)} concurrent forwards per step), each launch "
                                     "timed alone; in the loop the forwards overlap" if two_branch else "both CFG branches (2B rows) per launch"),
                    "note": ("algorithmic FLOPs (one product per MAC) over measured time; the split-bf16 arm spends %d tensor-core "
                             "products per MAC for fp32-level parity" % {0: 0, 1: 1, 2: 3, 3: 6}[SPLIT_TERMS])}
        if config3 is not None and SPLIT_TERMS == 2:
            # the same per-launch view at the launch shapes of configs[2] (the rows of this rank's share of the global batch 32)
            try:
                B3 = hi - lo
                model._cond_sig = None
                model.prepare(dict(y_dev3), B3, T, dev)
                x3 = torch.randn(B3, T, w["C"], device=dev)
                ts3 = torch.full((B3,), 500, device=dev, dtype=torch.int64)
                ws3 = model._workspace(lib.a2p_workspace_bytes(C.byref(model._cfg), B3, T), dev)
                g3 = int(lib.a2p_loop_row_groups(model._handle, B3, T))
                units3 = [(3, 0, B3)] if g3 == 0 else [(mk, B3 * g // g3, B3 * (g + 1) // g3 - B3 * g // g3) for g in range(g3) for mk in (1, 2)]
                acc3, cnt3 = np.zeros(ncat), np.zeros(ncat, dtype=np.int64)
                for i in range(4):
                    for mk, b0, bs in units3:
                        _lib.check(lib.a2p_profile_forward_rows(model._handle, B3, b0, bs, T, x3[b0:].data_ptr(), ts3[b0:].data_ptr(), mk,
                                                                ws3.data_ptr(), ws3.numel(), torch.cuda.current_stream().cuda_stream,
                                                                ms_cat, n_cat_c, ncat))
                        if i:
                            acc3 += np.array(list(ms_cat))
                        if i == 1:
                            cnt3 += np.array(list(n_cat_c), dtype=np.int64)
                acc3 /= 3
                R3 = 2 * B3
                alg3 = {4: 4 * T * (S + 2) * D * R3 * L / max(1, cnt3[4]), 3: 4 * T * T * D * R3 * L / max(1, cnt3[3]),
                        2: 8 * T * D * D * R3 * L / max(1, cnt3[2]), 6: (2 * T * D * D + 4 * T * D * 1024 + 6 * T * D * D) * R3 * L / max(1, cnt3[6])}
                per = {}
                for k_ in (4, 3, 6, 2):
                    msl = acc3[k_] / max(1, cnt3[k_])
                    tf = alg3[k_] / (msl * 1e-3) / 1e12 if msl > 0 else 0.0
                    per[names[k_]] = {"ms_per_launch": round(float(msl), 5), "achieved_tflops": round(float(tf), 2), "frac": round(float(tf / peak_tf), 4),
                                      "launches_per_forward": int(cnt3[k_])}
                config3["roofline_per_launch"] = {"rows_per_launch": units3[0][2], "concurrent_forwards": len(units3), "peak": peak_tf, "unit": "TFLOP/s",
                                                  "kernels": per, "note": "algorithmic FLOPs per launch / CUDA-event time of the launch timed alone, as in `roofline`"}
            except Exception as e:   # diagnostics only: never lose the contract line over it
                config3["roofline_per_launch"] = {"error": str(e)[:200]}
        gpu_base = None
        if not a.no_gpu_baseline and world == 1 and not face and not a.no_cfg:
            gpu_base = {"configs[1]": gpu_baseline(B)}
            if config3 is not None:
                gpu_base["configs[2]"] = gpu_baseline(CONFIG3_GLOBAL_BATCH)
                gb = gpu_base["configs[2]"]
                if gb and gb.get("value"):
                    config3["vs_gpu_baseline"] = config3["value"] / gb["value"]
        if not a.no_cpu_baseline and world == 1:      # reported on rank 0 at N = 1 only (the contract); the reference arm covers N > 1
            cpu_base = cpu_baseline(w["fmt"])
        f_fwd = flops_per_sample_forward(T=T, S=S + 2, S2=20, D=model.dims.D, L=L, FF=1024, C=w["C"], fmt=w["fmt"])
        if config3 is not None:
            config3["roofline_step_level"] = {"achieved": f_fwd * 2 * CONFIG3_GLOBAL_BATCH * n_diff / (config3["ms_per_step"] * 1e-3) / 1e12,
                                              "unit": "TFLOP/s"}
            config3["roofline_step_level"]["frac_of_sustained"] = config3["roofline_step_level"]["achieved"] / peaks.get("bf16_tflops_sustained", peak_tf)
        # whole-step view beside the per-launch one: the concurrent forwards share the machine, so the step as a whole sustains
        # more than any single launch timed alone
        step_tf = f_fwd * nbr * B * n_diff / (ms_step * 1e-3) / 1e12
        roofline["step_level"] = {"achieved": step_tf, "frac": step_tf / peak_tf,
                                  "frac_of_sustained": step_tf / peaks.get("bf16_tflops_sustained", peak_tf), "concurrent_forwards": len(units),
                                  "note": "algorithmic FLOPs of a whole loop / loop time on this GPU"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if SPLIT_TERMS == 0 else f"bf16x{SPLIT_TERMS} split (fp32-equivalent), fp32 accumulate",
            "data": "synthetic",
            "config": {"workload": workload_name(w["fmt"], B, not a.no_cfg, n_diff),
                       "global_batch": B * world, "parallelism": f"batch-sharded x{world}, 1 all-gather",
                       "l2": "inputs_larger_than_l2 (K/V caches %d MB + activations per step)" % (B * 25),
                       "algorithmic_gflop_per_loop": f_fwd * nbr * B * world * n_diff / 1e9},
            "clocks": clk, "gpu_launches": int(launches),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": ms_e2e},
            "roofline": roofline, "cpu_baseline": cpu_base, "gpu_baseline": gpu_base, "config3_strong": config3,
            "model_tflops": f_fwd * nbr * B * world * n_diff / (ms_step * 1e-3) / 1e12,
            "one_time": {"conditioning_ms": cond_ms, "share_of_loop": cond_ms / ms_step,
                         "what": "per distinct y, inside every timed loop: native conditioning encoders (cond_projection, pooled MLP, "
                                 "keyframe projection; a2p_denoiser_encode_conditioning) + per-layer rotated-K / V caches of both "
                                 "CFG branches (a2p_denoiser_set_conditioning), exact fp32"},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
