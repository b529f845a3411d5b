"""TEST INFRASTRUCTURE ONLY -- imports the *unmodified* reference from /root/reference.

Only usable where the reference tree is present (REFERENCE_ROOT); it is used by
oracle/make_golden.py and oracle/make_reference_units.py to record the reference's
outputs as tests/golden/*, which the tests compare against.  Nothing in the product
package may import this file.

Shims (SURVEY.md section 8c / Appendix B):
  * `azfuse`, `boto3`, `botocore` are absent -> stub packages in oracle/stubs
    (imported at generativeimage2text/torch_common.py:5, layers/bert/file_utils.py:19,21).
  * `clip.load` downloads weights (layers/CLIP/clip.py:64-83) -> replaced by a constructor of
    the same `VisualTransformer` that `build_model` would create
    (layers/CLIP/model.py:405-410: ViT-B/16 = (224,16,768,12,12,512), ViT-L/14 = (224,14,1024,24,16,768)).
  * the HF tokenizer needs a vocab download -> a stub carrying the two ids the model reads
    (generativeimage2text/model.py:35,54-55): cls=101, sep=102 (bert-base-uncased).
"""
import os
import sys

import torch

REFERENCE_ROOT = os.environ.get('GIT_REFERENCE_ROOT', '/root/reference')
_STUBS = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'stubs')

CLIP_CFG = {
    'ViT-B/16': dict(input_resolution=224, patch_size=16, width=768, layers=12, heads=12, output_dim=512),
    'ViT-L/14': dict(input_resolution=224, patch_size=14, width=1024, layers=24, heads=16, output_dim=768),
}


class Tok(object):
    cls_token_id = 101
    sep_token_id = 102


def reference_available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, 'generativeimage2text'))


def _import_reference():
    if not reference_available():
        raise RuntimeError('reference tree not present at %s' % REFERENCE_ROOT)
    for p in (REFERENCE_ROOT, _STUBS):
        if p not in sys.path:
            sys.path.insert(0, p)
    from generativeimage2text.layers.CLIP import clip
    from generativeimage2text.layers.CLIP.model import VisualTransformer

    class Holder(torch.nn.Module):
        def __init__(self, visual):
            super().__init__()
            self.visual = visual

    def fake_load(name, device='cpu', jit=False, **kw):
        return Holder(VisualTransformer(**CLIP_CFG[name])), None

    clip.load = fake_load
    import generativeimage2text.model as ref_model
    import generativeimage2text.layers.decoder as ref_decoder
    return ref_model, ref_decoder


def load_reference_model(param=None, search='greedy', max_steps=40, state_dict=None,
                         use_history=False):
    """Build the reference CaptioningModel (model.py:9-61) on CPU/fp32, eval mode.

    search: 'greedy' = the reference's commented-out greedy config (model.py:27-33),
            'beam'   = GeneratorWithBeamSearch(beam 4, lp 0.6) with max_steps lowered (model.py:34-40),
            'stock'  = leave the shipped decoder untouched.
    use_history: flip the dormant hidden-state cache on (SURVEY.md section 0 item 1) -- results-equivalent,
            4.5x faster on CPU; used only to cross-check.
    """
    ref_model, ref_decoder = _import_reference()
    param = dict(param or {})
    model = ref_model.get_git_model(Tok(), param)
    if search == 'greedy':
        model.decoder = ref_decoder.AutoRegressiveBeamSearch(
            eos_index=Tok.sep_token_id, max_steps=max_steps, beam_size=1,
            per_node_beam_size=1, fix_missing_prefix=True)
    elif search == 'beam':
        model.decoder = ref_decoder.GeneratorWithBeamSearch(
            eos_index=Tok.sep_token_id, max_steps=max_steps, beam_size=4, length_penalty=0.6)
    elif search != 'stock':
        raise ValueError(search)
    if state_dict is not None:
        missing, unexpected = model.load_state_dict(state_dict, strict=False)
        assert not unexpected, unexpected
        assert not [m for m in missing if not m.endswith('output.weight')], missing
    if use_history:
        model.textual.transformer.encoder.output_hidden_states = True
    model.eval()
    return model
