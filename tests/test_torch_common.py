"""Checkpoint ingestion (SURVEY.md section 8f-1): generativeimage2text_b200/torch_common.py against the reference's
torch_common.py (what it returned on the same inputs, stored under tests/golden) and against hand-checked cases."""
import collections

import pytest
import torch

from generativeimage2text_b200 import torch_common as tc
from generativeimage2text_b200.model import get_git_model
from generativeimage2text_b200.synthetic import synthetic_state_dict
from helpers import digest, load_golden


class Tok:
    cls_token_id, sep_token_id = 101, 102


def _messy_checkpoint(param, seed=3):
    """A checkpoint as training jobs leave them: DataParallel prefixes (twice on some keys), an extra optimizer-ish
    tensor, one tensor of the wrong shape, one tensor missing, short names that only match as suffixes."""
    sd = synthetic_state_dict(param, seed, 'perturbed')
    out = collections.OrderedDict()
    for i, (k, v) in enumerate(sd.items()):
        if k == 'textual.embedding.positions.weight':
            out['module.' + k] = v[:512].clone()            # wrong shape -> ignored, model keeps its own
        elif k == 'image_encoder.ln_post.bias':
            continue                                         # missing -> model keeps its own
        elif k.startswith('image_encoder.transformer.resblocks.3.'):
            out['module.module.' + k] = v                    # prefix twice
        elif k.startswith('textual.transformer.encoder.layer.2.'):
            out[k[len('textual.'):]] = v                     # only a suffix of the model key
        else:
            out['module.' + k] = v
    out['module.optimizer_step'] = torch.zeros(1)
    return out, sd


def test_prefix_and_suffix_rules():
    assert tc.remove_prefix({'module.module.a.b': 1, 'c': 2}, 'module.') == {'a.b': 1, 'c': 2}
    model_sd = {'x.layer.weight': 0, 'layer.weight': 0, 'y.bias': 0, 'lonely': 0}
    loaded = {'layer.weight': torch.zeros(1), 'weight': torch.ones(1), 'bias': torch.full((1,), 2.0)}
    tc.align_and_update_state_dicts(model_sd, loaded)
    # longest suffix wins; keys without any match are dropped from the dict that is then loaded
    assert set(model_sd) == {'x.layer.weight', 'layer.weight', 'y.bias'}
    assert model_sd['x.layer.weight'].item() == 0 and model_sd['layer.weight'].item() == 0 and model_sd['y.bias'].item() == 2


@pytest.mark.parametrize('param', [{}, {'num_image_with_embedding': 6}])
def test_load_state_dict_into_engine_shell(param):
    model = get_git_model(Tok(), param)
    before = {k: v.clone() for k, v in model.state_dict().items()}
    ckpt, sd = _messy_checkpoint(param)
    tc.load_state_dict(model, ckpt)
    after = model.state_dict()
    for k, v in sd.items():
        if k in ('textual.embedding.positions.weight', 'image_encoder.ln_post.bias'):
            assert torch.equal(after[k], before[k]), k       # skipped: shape mismatch / absent
        else:
            assert torch.equal(after[k], v), k
    assert after['textual.output.weight'].data_ptr() == after['textual.embedding.words.weight'].data_ptr()


def test_same_result_as_reference_loader():
    """Every tensor ends up where the reference's torch_common.load_state_dict puts it: the checkpoint key it took, or the
    model's own starting value (recorded by oracle/make_reference_units.py on the same checkpoint)."""
    g = load_golden('reference_torch_common')['meta']['loader']
    param = g['param']
    ckpt, _ = _messy_checkpoint(param, g['ckpt_seed'])
    ours = get_git_model(Tok(), param)
    # same starting point for the tensors the checkpoint does not provide
    start = synthetic_state_dict(param, g['start_seed'], 'init')
    ours.load_state_dict(start, strict=True)
    tc.load_state_dict(ours, ckpt)
    osd = ours.state_dict()
    assert list(osd.keys()) == [k for k, _ in g['source']]
    for k, src in g['source']:
        assert torch.equal(osd[k], start[k] if src is None else ckpt[src]), k


@pytest.mark.parametrize('patch,width,after', [(16, 768, 480), (14, 1024, 420), (16, 768, 160)])
def test_resize_2d_pos_embed_equals_reference(patch, width, after):
    """Bit for bit against the reference's resize_2d_pos_embed output (sha256 stored by oracle/make_reference_units.py)."""
    want = [c for c in load_golden('reference_torch_common')['meta']['pos_embed']
            if (c['patch'], c['width'], c['after']) == (patch, width, after)]
    assert len(want) == 1
    want = want[0]
    g = 224 // patch
    pe = torch.randn(g * g + 1, width, generator=torch.Generator().manual_seed(5))
    b = tc.resize_2d_pos_embed(pe, 224, patch, after)
    assert list(b.shape) == want['shape'] == [(after // patch) ** 2 + 1, width]
    assert digest(b) == want['sha256']
    b3 = tc.resize_2d_pos_embed(pe[None], 224, patch, after)
    assert list(b3.shape) == want['shape_batched'] and digest(b3) == want['sha256_batched']
