"""Shared helpers for the parity tests (test infrastructure)."""
import hashlib
import json
import os

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
SAMPLE_STRIDE = 1021     # strided sample kept beside a digest where a full array would not fit a golden file


def load_golden(name):
    g = np.load(os.path.join(GOLDEN_DIR, name + '.npz'))
    d = {k: g[k] for k in g.files}
    d['meta'] = json.loads(str(d['meta']))
    return d


def digest(a):
    """sha256 of an array's values in C order (with its dtype): bit-exact comparison against a stored reference output."""
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    return hashlib.sha256(a.dtype.str.encode() + np.ascontiguousarray(a).tobytes()).hexdigest()


def strided_sample(a):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    return np.ascontiguousarray(a).reshape(-1)[::SAMPLE_STRIDE].copy()


def golden_inputs(meta):
    from generativeimage2text_b200.synthetic import synthetic_state_dict, synthetic_images
    sd = synthetic_state_dict(meta['param'], meta['seed'], meta['variant'])
    image = synthetic_images(meta['batch'], meta['frames'], meta['img_seed'], meta.get('image_hw', 224))
    batch = {'image': image}
    if 'prefix' in meta:
        batch['prefix'] = torch.tensor([meta['prefix']], dtype=torch.long)
    return sd, batch


def greedy_margins(raw_logits, tokens_in, eos=102):
    """Decision margin (top1 - top2) per row of one greedy step after the reference's masking
    (no-repeat scatter, layers/decoder.py:330; skipped on the very first step :257-273)."""
    z = raw_logits.clone()
    if tokens_in is not None:
        z.scatter_(1, tokens_in[:, None], -10000.0)
    top = z.topk(2, dim=1).values
    return top[:, 0] - top[:, 1]


def golden_greedy_margins(g, i, tokens_in):
    """The same margin from what a golden file stores (the reference's top-4 raw logits per row and step): the no-repeat
    scatter removes the input token from the ranking (never on the first step)."""
    vals, idx = g['step_top4_val'][i], g['step_top4_idx'][i]
    out = np.zeros(vals.shape[0], dtype=np.float64)
    for r in range(vals.shape[0]):
        keep = [v for v, t in zip(vals[r], idx[r]) if tokens_in is None or t != int(tokens_in[r])]
        out[r] = keep[0] - keep[1]
    return out
