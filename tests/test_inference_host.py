"""CPU: host logic of generativeimage2text_b200/inference.py -- the size rules of the image transform against the
oracle (itself pinned to PIL / torchvision / the reference in tests/test_preprocess_oracle.py), the weight tables the
library builds on the host against the oracle's, and the no-CPU-path guarantee of the transform."""
import ctypes

import numpy as np
import pytest
import torch

import preprocess_oracle as po
from helpers import load_golden
from generativeimage2text_b200 import inference as inf
from generativeimage2text_b200 import _lib

SHAPES = [(480, 640), (640, 480), (224, 224), (225, 1000), (37, 41), (1000, 225), (300, 224), (612, 408), (97, 301),
          (420, 420), (480, 480), (1, 9), (3000, 2000)]


@pytest.mark.parametrize('param', [{}, {'test_crop_size': 160}, {'test_crop_size': 480, 'test_respect_ratio_max': 640},
                                   {'test_crop_size': 420, 'test_respect_ratio_max': 560}])
def test_geometry_equals_oracle_rules(param):
    t = inf.ImageTransform(param, device='cpu')
    crop = param.get('test_crop_size', 224)
    for h, w in SHAPES:
        rh, rw, top, left, oh, ow = t.geometry(h, w)
        if 'test_respect_ratio_max' in param:
            assert (rh, rw) == (oh, ow) == po.minmax_size(h, w, crop, param['test_respect_ratio_max'])
            assert (top, left) == (0, 0)
        else:
            assert (rh, rw) == po.resize_shorter_edge(h, w, crop)
            assert (top, left) == po.center_crop_box(rh, rw, crop)
            assert (oh, ow) == (crop, crop)


def test_minmax_equals_reference_class():
    """Sizes and repr against what the reference's MinMaxResizeForTest returned (stored by oracle/make_reference_units.py)."""
    g = load_golden('reference_transform')['meta']['minmax']
    assert [(c['min'], c['max']) for c in g] == [(480, 640), (420, 560), (224, 224)]
    for c in g:
        b = inf.MinMaxResizeForTest(c['min'], c['max'])
        assert [s[:2] for s in c['sizes']] == [list(hw) for hw in SHAPES]
        for h, w, want in c['sizes']:
            assert list(b.get_size((w, h))) == want
        assert repr(b) == c['repr']


@pytest.mark.parametrize('pair', [(640, 298), (480, 224), (75, 224), (500, 720), (1920, 398), (3, 2), (5, 7), (224, 112),
                                  (333, 480), (1, 5), (7, 1), (4000, 224), (223, 224), (224, 224)])
def test_library_weight_tables_equal_oracle(pair):
    """gitb200_preproc_coeffs (host code of the library, no GPU needed) == Resample.c's tables as restated by the oracle."""
    lib = _lib.load()
    a, b = pair
    ks = ctypes.c_int32()
    assert lib.gitb200_preproc_coeffs(a, b, ctypes.byref(ks), None, None, 0) == 0
    if a == b:
        assert ks.value == 1        # identity window: Pillow skips the pass
        return
    k, bounds, kk = po.precompute_coeffs(a, b)
    assert ks.value == k
    B = np.zeros((b, 2), np.int32)
    K = np.zeros((b, k), np.int32)
    assert lib.gitb200_preproc_coeffs(a, b, ctypes.byref(ks), B.ctypes.data, K.ctypes.data, k) == 0
    assert np.array_equal(B, bounds) and np.array_equal(K, kk)
    assert lib.gitb200_preproc_coeffs(a, b, ctypes.byref(ks), B.ctypes.data, K.ctypes.data, k - 1) != 0   # too small


def test_transform_has_no_cpu_path():
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    t = inf.get_image_transform({})
    with pytest.raises(RuntimeError):
        t(np.zeros((32, 32, 3), dtype=np.uint8))
    h = ctypes.c_void_p()
    assert _lib.load().gitb200_preproc_create(0, ctypes.byref(h)) != 0


def test_row_formats():
    assert inf.json_dump([{'caption': 'a b'}]) == '[{"caption":"a b"}]'
    assert inf.json_dump({'question_id': 3, 'answer': 'x'}) == '{"answer":"x","question_id":3}'
    assert inf.pilimg_from_base64('!!!not base64!!!') is None


def test_yaml_base_is_merged_per_path(tmp_path):
    """`_base_` files are merged path by path like the reference's load_from_yaml_file (tsv_io.py:97-107): a child that
    overrides one nested key keeps the rest of the base's sub-dictionary."""
    from generativeimage2text_b200.inference import load_from_yaml_file
    (tmp_path / 'base.yaml').write_text('param:\n  a: 1\n  b: {c: 2, d: 3}\nname: base\nlst: [1, 2]\n')
    (tmp_path / 'child.yaml').write_text('_base_: base.yaml\nparam:\n  b: {c: 20}\nlst: [9]\n')
    got = load_from_yaml_file(str(tmp_path / 'child.yaml'))
    assert got == {'param': {'a': 1, 'b': {'c': 20, 'd': 3}}, 'name': 'base', 'lst': [9]}


def test_respect_ratio_key_presence_selects_the_transform():
    """The reference tests `'test_respect_ratio_max' in param` (inference.py:113), not the value's truthiness."""
    from generativeimage2text_b200.inference import ImageTransform
    assert ImageTransform({'test_crop_size': 160}, device='cpu').minmax is None
    assert ImageTransform({'test_crop_size': 160, 'test_respect_ratio_max': 224}, device='cpu').minmax is not None
    assert ImageTransform({'test_crop_size': 160, 'test_respect_ratio_max': 0}, device='cpu').minmax is not None
