"""Shared by make_golden.py (run where /root/reference exists) and the tests (run anywhere):
deterministic synthetic weights / clips so fixtures only need to store OUTPUTS."""
import hashlib

import torch

C1 = dict(model_name='vit_tiny', crop_size=224, patch_size=16, num_frames=8, tubelet_size=2, batch=2,
          pred_depth=12, pred_embed_dim=384, depth=12, heads=3, embed_dim=192)

VITL16_MASKS = [
    dict(aspect_ratio=[0.75, 1.5], num_blocks=8, spatial_scale=[0.15, 0.15], temporal_scale=[1.0, 1.0],
         max_temporal_keep=1.0, max_keep=None),
    dict(aspect_ratio=[0.75, 1.5], num_blocks=2, spatial_scale=[0.7, 0.7], temporal_scale=[1.0, 1.0],
         max_temporal_keep=1.0, max_keep=None),
]


def sha16(t):
    return hashlib.sha256(t.contiguous().numpy().tobytes()).hexdigest()[:16]


def synth_state(shapes, seed, keep=()):
    """name -> tensor, values from a seeded CPU generator in sorted-name order (stable across machines)."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for name in sorted(shapes):
        shape = tuple(shapes[name])
        if any(name.endswith(k) for k in keep):
            continue
        r = torch.randn(shape, generator=g)
        if name.endswith('bias'):
            out[name] = 0.02 * r
        elif 'norm' in name and name.endswith('weight'):
            out[name] = 1.0 + 0.1 * r
        elif 'mask_tokens' in name:
            out[name] = 0.02 * r
        else:
            out[name] = 0.03 * r
    return out


def synth_clips(B, T, H, W, seed=0):
    return torch.randn(B, 3, T, H, W, generator=torch.Generator().manual_seed(seed))


def sample_index(numel, n):
    """At most n flat indices spread over a tensor of numel elements (golden-ratio sequence: no RNG, identical on
    every machine and torch version); every index when numel <= n.  Fixtures store values at these positions only."""
    if numel <= n:
        return torch.arange(numel)
    j = torch.arange(n, dtype=torch.float64)
    return (torch.remainder(j * 0.6180339887498949, 1.0) * numel).long()
