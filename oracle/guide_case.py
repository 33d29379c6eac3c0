"""TEST INFRASTRUCTURE: the inputs of the guide-sampler and VQ-decoder parity cases (tests/test_guide.py).

The reference's GuideTransformer (model/guide.py) and TemporalVertexCodec (model/vqvae.py) are run once on CPU by
oracle/make_golden.py guide with the weights built here; tests/golden/guide.npz keeps their outputs, the checkpoint layout
(key, shape, dtype of every entry) and the few buffers whose values are fixed by construction (rotary frequencies,
resampling kernel).  Every other weight is regenerated from a seed on both sides, so the golden file stays small."""
from __future__ import annotations

import json
import math

import torch

GUIDE = dict(tokens=32, layers=2, dim=64, B=2, n=12, seed=5)
VQ = dict(n_vertices=104, latent_dim=64, categories=32, residual_depth=4, seed=2)


def layout(state_dict) -> str:
    """JSON list of [key, shape, dtype] in state_dict order"""
    return json.dumps([[k, list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in state_dict.items()])


def seeded_state(layout_json: str, seed: int, fixed=None):
    """weights for `layout_json`: `fixed` entries as given; other float entries N(0, 1/(3 fan_in)), the spread of PyTorch's
    default Linear / Conv initialisation, and N(0, 0.05^2) for vectors, so every bias and affine term is non-trivial;
    integer / bool entries ones (the codebooks' `inited` flags)."""
    fixed = fixed or {}
    g = torch.Generator().manual_seed(seed)
    out = {}
    for name, shape, dtype in json.loads(layout_json):
        dt = getattr(torch, dtype)
        if name in fixed:
            out[name] = torch.as_tensor(fixed[name]).to(dt).reshape(shape)
        elif dt.is_floating_point:
            std = 0.05 if len(shape) <= 1 else (3 * math.prod(shape[1:])) ** -0.5
            out[name] = (torch.randn(shape, generator=g) * std).to(dt)
        else:
            out[name] = torch.ones(shape, dtype=dt)
    return out


def guide_audio(B: int, frames: int = 240, seed: int = 3):
    g = torch.Generator().manual_seed(seed)
    return 0.1 * torch.randn(B, frames * 1600, 2, generator=g)


def guide_tokens(B: int, n: int, tokens: int, seed: int = 9):
    """a start token followed by random codes"""
    g = torch.Generator().manual_seed(seed)
    return torch.cat([torch.full((B, 1), tokens), torch.randint(0, tokens, (B, n - 1), generator=g)], dim=1)


def uniform_tape(B: int, seed: int = 11):
    return torch.rand(64, B, generator=torch.Generator().manual_seed(seed))


def inverse_cdf_draw(tape):
    """categorical draw from `probs` through the next row of `tape` (the same draw on both sides)"""
    it = iter(tape)
    return lambda probs: (torch.cumsum(probs, -1) < next(it).unsqueeze(-1)).sum(-1).clamp(max=probs.shape[-1] - 1)


def vq_codes(seed: int = 4):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, VQ["categories"], (3, 20, VQ["residual_depth"]), generator=g)
