"""TEST INFRASTRUCTURE ONLY -- imports the unmodified reference from /root/reference.

This module exists only in the build container (the GPU box has no /root/reference); it is
used by oracle/make_golden.py to (a) pin oracle/a2p_oracle.py against the running reference
and (b) emit the golden fixtures committed under tests/golden/.  Nothing in the product
package imports it.

Shims (harness-side only, /root/reference is never edited) -- SURVEY.md section 8c:
  1. stand-in `fairseq` module (fairseq==0.12.2 is pinned by demo/requirements.txt:3 but is not
     installed/vendored): `checkpoint_utils.load_model_ensemble_and_task` returns a random-init
     module exposing `feature_extractor` / `feature_aggregator` with the published conv geometry
     (model/utils.py:19-21, model/modules/audio_encoder.py:28-31).
  2. pose on CPU: `Tensor.cuda()` neutralised (model/diffusion.py:321 hard-codes .cuda()).
  3. face: a fabricated ./assets/iter-0200000.pt in a scratch cwd (model/diffusion.py:273-277).
  4. `p_sample` repair (diffusion/gaussian_diffusion.py:476 uses an undefined `noise`): the two
     upstream-MDM lines are re-inserted by monkey-patch for the ancestral oracle.
The frozen audio encoders are OUTSIDE the replaced path: `encode_audio`/`encode_lip` are
bypassed so both sides consume the same synthetic wav2vec features (BASELINE config 2).
"""
from __future__ import annotations

import contextlib
import os
import sys
import tempfile
import types
from argparse import Namespace

import torch
import torch.nn as nn

_HERE = os.path.dirname(os.path.abspath(__file__))
# the reference tree itself in the build container; on the GPU box the pruned byte-for-byte view that
# oracle/build_ref.py wrote into oracle/_ref (git-ignored, travels with the snapshot)
REF_ROOT = "/root/reference" if os.path.isdir("/root/reference/diffusion") and not os.environ.get("A2P_FORCE_REF_VIEW") \
    else os.path.join(_HERE, "_ref")


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REF_ROOT, "diffusion"))


class _ConvStack(nn.Module):
    def __init__(self, layers):
        super().__init__()
        self.conv_layers = nn.ModuleList()
        cin = 1
        for dim, k, s in layers:
            self.conv_layers.append(
                nn.Sequential(nn.Conv1d(cin, dim, k, stride=s, bias=False), nn.Dropout(0.0),
                              nn.GroupNorm(1, dim), nn.ReLU())
            )
            cin = dim

    def forward(self, x):
        x = x.unsqueeze(1)
        for conv in self.conv_layers:
            x = conv(x)
        return torch.log(torch.abs(x) + 1)


class _StandInWav2Vec(nn.Module):
    def __init__(self, large: bool):
        super().__init__()
        if large:
            geo = [(512, 10, 5), (512, 8, 4), (512, 4, 2), (512, 4, 2), (512, 4, 2), (512, 1, 1), (512, 1, 1)]
        else:
            geo = [(512, 10, 5), (512, 8, 4), (512, 4, 2), (512, 4, 2), (512, 4, 2), (512, 1, 1), (512, 1, 1), (512, 1, 1)]
        self.feature_extractor = _ConvStack(geo)
        self.feature_aggregator = nn.Conv1d(512, 512, 1)


def fairseq_standin_modules() -> dict:
    """{import name: module} of the stand-in `fairseq` (shim 1)"""
    fs = types.ModuleType("fairseq")
    cu = types.ModuleType("fairseq.checkpoint_utils")

    def load_model_ensemble_and_task(paths, *a, **k):
        large = "large" in os.path.basename(paths[0])
        return [_StandInWav2Vec(large)], None, None

    cu.load_model_ensemble_and_task = load_model_ensemble_and_task
    fs.checkpoint_utils = cu
    return {"fairseq": fs, "fairseq.checkpoint_utils": cu}


def _install_fairseq_standin() -> None:
    if "fairseq" in sys.modules:
        return
    sys.modules.update(fairseq_standin_modules())


_scratch = None


def import_reference():
    """Put /root/reference on sys.path (read-only) and return the modules the path touches."""
    global _scratch
    assert reference_available(), "reference tree not present (this only runs in the build container)"
    _install_fairseq_standin()
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    if _scratch is None:
        _scratch = tempfile.mkdtemp(prefix="a2p_ref_")
        os.makedirs(os.path.join(_scratch, "assets"), exist_ok=True)
    import diffusion.gaussian_diffusion as gd  # noqa
    import diffusion.respace as respace  # noqa
    import model.diffusion as mdiff  # noqa
    import model.cfg_sampler as cfg  # noqa
    import utils.model_util as model_util  # noqa
    return Namespace(gd=gd, respace=respace, mdiff=mdiff, cfg=cfg, model_util=model_util, scratch=_scratch)


@contextlib.contextmanager
def _cwd(path):
    old = os.getcwd()
    os.chdir(path)
    try:
        yield
    finally:
        os.chdir(old)


def make_args(data_format: str, layers: int, heads: int, timestep_respacing: str, max_seq_length: int = 600,
              device="cpu", **extra) -> Namespace:
    return Namespace(
        data_format=data_format, add_frame_cond=1 if data_format == "pose" else None,
        max_seq_length=max_seq_length, layers=layers, heads=heads, not_rotary=False, unconstrained=False,
        device=device, timestep_respacing=timestep_respacing, noise_schedule="cosine", sigma_small=True,
        lambda_vel=0.0, model_path="synthetic/model.pt", resume_trans=None, **extra,
    )


def build_reference(data_format: str, layers: int, heads: int, timestep_respacing: str, state_dict=None, device="cpu"):
    """create_model_and_diffusion (utils/model_util.py:41-46) + load_model + CFG wrapper (CPU unless `device` says cuda)."""
    ref = import_reference()
    args = make_args(data_format, layers, heads, timestep_respacing, device=device)
    with _cwd(ref.scratch):
        if data_format == "face":
            lip_path = os.path.join(ref.scratch, "assets", "iter-0200000.pt")
            if not os.path.exists(lip_path):
                lip = ref.mdiff.Audio2LipRegressionTransformer()
                torch.save({"model_state_dict": lip.state_dict()}, lip_path)
        model, diffusion = ref.model_util.create_model_and_diffusion(args, split_type="test")
    if state_dict is not None:
        # real checkpoints carry the frozen fairseq modules too (load_model only tolerates missing
        # transformer./tokenizer. keys, utils/model_util.py:33-38): keep the stand-in's own values.
        full = {k: v for k, v in model.state_dict().items() if k.startswith(("audio_model.", "lip_model."))}
        full.update(state_dict)
        ref.model_util.load_model(model, full)
    model.eval()
    return ref, args, model, diffusion


@contextlib.contextmanager
def synthetic_features(model, feats: torch.Tensor):
    """Bypass the frozen encoders: encode_audio -> feats (pose [B,S,1024] / face [B,S,2038])."""
    cls = type(model)
    old_a, old_l = cls.encode_audio, cls.encode_lip
    cls.encode_audio = lambda self, raw: feats.to(raw.device)
    cls.encode_lip = lambda self, audio, cond_embed: cond_embed
    old_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self  # shim 2 (CPU oracle only)
    try:
        yield
    finally:
        cls.encode_audio, cls.encode_lip = old_a, old_l
        torch.Tensor.cuda = old_cuda


@contextlib.contextmanager
def repaired_p_sample(gd, noise_tape=None):
    """Shim 4: upstream-MDM `noise = th.randn_like(x)` (+ const_noise) re-inserted before :476.

    If `noise_tape` (list of tensors, consumed in call order) is given it replaces randn_like so
    that CPU oracle and CUDA path see the same per-step noise.
    """
    th = torch
    tape = list(noise_tape) if noise_tape is not None else None

    def p_sample(self, model, x, t, clip_denoised=True, denoised_fn=None, cond_fn=None, model_kwargs=None,
                 const_noise=False):
        out = self.p_mean_variance(model, x, t, clip_denoised=clip_denoised, denoised_fn=denoised_fn,
                                   model_kwargs=model_kwargs)
        noise = tape.pop(0) if tape is not None else th.randn_like(x)
        if const_noise:
            noise = noise[[0]].repeat(x.shape[0], 1, 1, 1)
        nonzero_mask = (t != 0).float().view(-1, *([1] * (len(x.shape) - 1)))
        sample = out["mean"] + nonzero_mask * th.exp(0.5 * out["log_variance"]) * noise
        return {"sample": sample, "pred_xstart": out["pred_xstart"]}

    old = gd.GaussianDiffusion.p_sample
    gd.GaussianDiffusion.p_sample = p_sample
    try:
        yield
    finally:
        gd.GaussianDiffusion.p_sample = old
