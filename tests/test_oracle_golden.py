"""CPU: oracle/git_oracle.py against the golden vectors produced by the unmodified reference
(oracle/make_golden.py); with tests/test_oracle_vs_reference.py, this pins the oracle on every machine."""
import numpy as np
import pytest
import torch

import git_oracle
from helpers import load_golden, golden_inputs

CASES = ['base_greedy_init', 'base_greedy', 'base_beam', 'base_prefix', 'vatex_greedy',
         'large_greedy', 'large_beam', 'base_ratio_greedy', 'base_crop160_greedy', 'base_vqa_ratio_greedy',
         # round 2: the benchmarked configurations at their benchmarked batch sizes, and the decisive-margin checkpoint
         'base_greedy_b64', 'vatex_greedy_b16', 'large_beam_b32', 'base_decisive']


@pytest.mark.parametrize('name', CASES)
def test_oracle_matches_reference_golden(name):
    g = load_golden(name)
    meta = g['meta']
    sd, batch = golden_inputs(meta)
    raw, taps = [], {}
    out = git_oracle.generate(sd, meta['param'], batch, meta['search'], meta['max_steps'],
                              cached=True, raw_trace=raw, taps=taps)
    # image features and visual projection (fp32 vs fp32: only op-order noise)
    np.testing.assert_allclose(taps['visual_features'][:, ::17, ::29].numpy(), g['feats_sample'],
                               rtol=0, atol=2e-4)
    np.testing.assert_allclose(taps['visual_projection'][:, ::17, ::29].numpy(), g['vproj_sample'],
                               rtol=0, atol=2e-4)
    # search result: token-identical, logprobs to fp32 noise
    assert out['predictions'].shape == tuple(g['predictions'].shape)
    assert np.array_equal(out['predictions'].numpy(), g['predictions'])
    np.testing.assert_allclose(out['logprobs'].numpy(), g['logprobs'], rtol=0, atol=2e-3)
    # every decoding_step call: sampled logits + top-2
    assert len(raw) == g['step_logits'].shape[0]
    cols = torch.from_numpy(g['vocab_cols'])
    for i, z in enumerate(raw):
        np.testing.assert_allclose(z[:, cols].numpy(), g['step_logits'][i], rtol=0, atol=5e-4)
        top = z.topk(2, dim=1)
        np.testing.assert_allclose(top.values.numpy(), g['step_top2_val'][i], rtol=0, atol=5e-4)


def test_as_shipped_equals_cached():
    """The shipped no-cache path and the KV-cached path are results-equivalent (SURVEY section 0 item 1)."""
    g = load_golden('base_greedy')
    meta = dict(g['meta'])
    meta['batch'] = 1
    sd, batch = golden_inputs(meta)
    a = git_oracle.generate(sd, meta['param'], batch, 'greedy', 12, cached=True)
    b = git_oracle.generate(sd, meta['param'], batch, 'greedy', 12, cached=False)
    assert torch.equal(a['predictions'], b['predictions'])
    assert torch.allclose(a['logprobs'], b['logprobs'], atol=1e-4)
    assert np.array_equal(a['predictions'].numpy()[0], g['predictions'][0, :12])
