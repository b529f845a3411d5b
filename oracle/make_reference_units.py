"""TEST INFRASTRUCTURE ONLY -- records what the UNMODIFIED reference's host-side units return on the inputs the CPU tests
use, as tests/golden/reference_*.npz, so that the comparisons with the reference run on every machine.

Run where the reference tree is present (oracle/ref_shim.py):  python oracle/make_reference_units.py [name ...]

  reference_tsv_io        tsv_io.py: writer output (.tsv / .lineidx / .lineidx.8b), reader rows, concat_tsv_files output
                          (tests/test_tsv_io.py)
  reference_transform     inference.py: get_image_transform output (shape, sha256 of the float32 planes, strided sample)
                          and MinMaxResizeForTest sizes / repr (tests/test_preprocess_oracle.py, tests/test_inference_host.py)
  reference_torch_common  torch_common.py: where load_state_dict takes every model tensor from (a checkpoint key or the
                          model's own value), resize_2d_pos_embed output digests (tests/test_torch_common.py)
  reference_model         model.py / layers/decoder.py / trie_decoder.py: state-dict layout and tied tensors, greedy and beam
                          captions on a seed outside tests/golden, trie-constrained and sampled searches on toy logits
                          (tests/test_oracle_vs_reference.py)

The inputs come from the test modules themselves, so a test and its golden file cannot drift apart.
"""
import json
import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
TESTS = os.path.join(ROOT, 'tests')
for p in (TESTS, HERE, ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import ref_shim  # noqa: E402
from helpers import GOLDEN_DIR, digest, strided_sample  # noqa: E402

TRANSFORM_PARAMS = [{}, {'test_crop_size': 480, 'test_respect_ratio_max': 640}]
TRANSFORM_SHAPES = [(480, 640), (1000, 300), (200, 200), (300, 1000), (480, 600)]
MINMAX_PAIRS = [(480, 640), (420, 560), (224, 224)]
POS_EMBED_CASES = [(16, 768, 480), (14, 1024, 420), (16, 768, 160)]


def save(name, meta, **arrays):
    meta = dict(meta, generator='oracle/make_reference_units.py', reference_commit='faae4fb9', torch=torch.__version__,
                numpy=np.__version__, cpu_capability=torch.backends.cpu.get_cpu_capability())
    path = os.path.join(GOLDEN_DIR, name + '.npz')
    np.savez_compressed(path, meta=np.array(json.dumps(meta)), **arrays)
    print('%-24s %7d bytes' % (name, os.path.getsize(path)))


def read_bytes(path):
    with open(path, 'rb') as fp:
        return np.frombuffer(fp.read(), dtype=np.uint8)


def reference_tsv_io():
    ref_shim._import_reference()
    import generativeimage2text.tsv_io as rio
    from test_tsv_io import _rows, _files
    rows = _rows(23, 7)
    arrays = {}
    with tempfile.TemporaryDirectory() as tmp:
        b = os.path.join(tmp, 'ref.tsv')
        rio.tsv_writer(iter(rows), b)
        for ext, f in zip(('tsv', 'lineidx', 'lineidx_8b'), _files(b)):
            arrays['written_' + ext] = read_bytes(f)
        t = rio.TSVFile(b)
        reads = {str(i): {'row': t[i], 'key': t.get_key(i)} for i in (0, 22, 9)}
        # merged parts; the reference's process pool is bypassed (num_worker=0)
        p1, p2 = os.path.join(tmp, 'p.0.2.tsv'), os.path.join(tmp, 'p.1.2.tsv')
        rio.tsv_writer(iter(rows[:10]), p1)
        rio.tsv_writer(iter(rows[10:]), p2)
        o = os.path.join(tmp, 'm_ref.tsv')
        orig = rio.parallel_map
        rio.parallel_map = lambda f, tasks, num_worker=0: [f(x) for x in tasks]
        os.environ['GIT_TMP_FOLDER'] = os.path.join(tmp, 'tmp')
        os.makedirs(os.path.join(os.environ['GIT_TMP_FOLDER'], tmp.lstrip('/')), exist_ok=True)
        try:
            rio.concat_tsv_files([p1, p2], o)
        finally:
            rio.parallel_map = orig
        arrays['merged_tsv'] = read_bytes(o)
        arrays['merged_lineidx_8b'] = read_bytes(_files(o)[2])
    save('reference_tsv_io', {'rows': [23, 7], 'split': 10, 'reads': reads}, **arrays)


def reference_transform():
    ref_shim._import_reference()
    import generativeimage2text.inference as rinf
    from PIL import Image
    from test_preprocess_oracle import _img
    from test_inference_host import SHAPES
    transform, arrays = [], {}
    for param in TRANSFORM_PARAMS:
        t = rinf.get_image_transform(param)
        for hw in TRANSFORM_SHAPES:
            want = t(Image.fromarray(_img(hw[0], hw[1], 3))).numpy()
            case = {'param': param, 'hw': list(hw), 'img_seed': 3, 'shape': list(want.shape), 'sha256': digest(want)}
            if 'test_respect_ratio_max' in param:
                mm = rinf.MinMaxResizeForTest(param['test_crop_size'], param['test_respect_ratio_max'])
                case['minmax_size'] = list(mm.get_size((hw[1], hw[0])))
            arrays['transform_%d_sample' % len(transform)] = strided_sample(want)
            transform.append(case)
    minmax = []
    for mn, mx in MINMAX_PAIRS:
        a = rinf.MinMaxResizeForTest(mn, mx)
        minmax.append({'min': mn, 'max': mx, 'repr': repr(a),
                       'sizes': [[h, w, list(a.get_size((w, h)))] for h, w in SHAPES]})
    save('reference_transform', {'transform': transform, 'minmax': minmax}, **arrays)


def reference_torch_common():
    ref_shim._import_reference()
    import generativeimage2text.torch_common as rtc
    from generativeimage2text_b200.synthetic import synthetic_state_dict
    from test_torch_common import _messy_checkpoint
    param = {'num_image_with_embedding': 6}
    ckpt, _ = _messy_checkpoint(param)
    ref = ref_shim.load_reference_model(param, 'stock')
    start = synthetic_state_dict(param, 11, 'init')
    ref.load_state_dict(start, strict=False)
    rtc.load_state_dict(ref, ckpt)
    by_digest = {}
    for k, v in ckpt.items():
        by_digest.setdefault(digest(v), k)
    source = []
    for k, v in ref.state_dict().items():
        d = digest(v)
        if d in by_digest:
            source.append([k, by_digest[d]])
        else:
            assert torch.equal(v, start[k]), 'tensor %s comes from neither the checkpoint nor the starting model' % k
            source.append([k, None])
    pos = []
    for patch, width, after in POS_EMBED_CASES:
        g = 224 // patch
        pe = torch.randn(g * g + 1, width, generator=torch.Generator().manual_seed(5))
        a = rtc.resize_2d_pos_embed(pe, 224, patch, after)
        a3 = rtc.resize_2d_pos_embed(pe[None], 224, patch, after)
        pos.append({'patch': patch, 'width': width, 'after': after, 'shape': list(a.shape), 'sha256': digest(a),
                    'shape_batched': list(a3.shape), 'sha256_batched': digest(a3)})
    save('reference_torch_common', {'loader': {'param': param, 'ckpt_seed': 3, 'start_seed': 11, 'source': source},
                                    'pos_embed': pos})


def reference_model():
    import git_oracle
    from generativeimage2text_b200.synthetic import synthetic_state_dict, synthetic_images
    from test_oracle_vs_reference import _toy_step, _toy_trie_sequences
    _, ref_decoder = ref_shim._import_reference()
    import generativeimage2text.trie_decoder as td
    layout = []
    for param in ({}, {'num_image_with_embedding': 6}):
        rsd = ref_shim.load_reference_model(param, 'greedy', 40).state_dict()
        groups = {}
        for k, v in rsd.items():
            groups.setdefault(v.data_ptr(), []).append(k)
        layout.append({'param': param, 'keys': [[k, list(v.shape)] for k, v in rsd.items()],
                       'tied': [g for g in groups.values() if len(g) > 1]})
    arrays = {}
    # a seed / image set that is not in tests/golden
    sd = synthetic_state_dict({}, seed=7, variant='init')
    img = synthetic_images(1, 0, seed=99)
    for search in ('greedy', 'beam'):
        with torch.no_grad():
            r = ref_shim.load_reference_model({}, search, 10, state_dict=sd)({'image': img})
        arrays['fresh_%s_predictions' % search] = r['predictions'].numpy()
        arrays['fresh_%s_logprobs' % search] = r['logprobs'].numpy()
    # TrieAutoRegressiveBeamSearch at batch 1 (the case that decoder supports)
    eos, start = 2, torch.tensor([[1]])
    for seed in range(4):
        dec = td.TrieAutoRegressiveBeamSearch(eos, max_steps=12, beam_size=1, trie=td.TokenTrie.construct(_toy_trie_sequences(eos)))
        rp, rl = dec.search(start, _toy_step(seed=seed))
        arrays['trie_%d_predictions' % seed], arrays['trie_%d_logprobs' % seed] = rp.numpy(), rl.numpy()
    # the do_sample branches of AutoRegressiveBeamSearch with torch.multinomial replaced by the inverse-CDF draw
    B, steps = 4, 14
    start = torch.tensor([[1]] * B)
    u = torch.rand((steps, B), generator=torch.Generator().manual_seed(5))
    for temperature in (1.0, 0.7):
        for seed in range(3):
            dec = ref_decoder.AutoRegressiveBeamSearch(eos, max_steps=steps, beam_size=1, per_node_beam_size=1,
                                                       fix_missing_prefix=True)
            calls = {'t': start.shape[1]}

            def fake_multinomial(probs, num_samples):
                assert num_samples == 1
                t = calls['t']
                calls['t'] += 1
                return git_oracle.inverse_cdf_draw(probs, u[t])[:, None]
            real = torch.multinomial
            torch.multinomial = fake_multinomial
            try:
                rp, rl = dec.search(start, _toy_step(seed=seed), do_sample=True, temperature=temperature)
            finally:
                torch.multinomial = real
            arrays['sample_%g_%d_predictions' % (temperature, seed)] = rp.numpy()
            arrays['sample_%g_%d_logprobs' % (temperature, seed)] = rl.numpy()
    save('reference_model', {'layout': layout, 'fresh': {'weight_seed': 7, 'variant': 'init', 'img_seed': 99, 'max_steps': 10},
                             'trie_seeds': 4, 'sample_seeds': 3}, **arrays)


UNITS = {f.__name__: f for f in (reference_tsv_io, reference_transform, reference_torch_common, reference_model)}

if __name__ == '__main__':
    if not ref_shim.reference_available():
        sys.exit('reference tree not found at %s (set GIT_REFERENCE_ROOT)' % ref_shim.REFERENCE_ROOT)
    for n in sys.argv[1:] or list(UNITS):
        UNITS[n]()
