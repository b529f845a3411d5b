"""Pins oracle/preprocess_oracle.py (the CPU restatement of the reference's test-time transform, SURVEY.md section
8f-2) against the third-party code the reference actually calls -- Pillow's resize and torchvision's transforms,
executing here -- bit for bit; and against what the reference's own `get_image_transform` / `MinMaxResizeForTest`
returned."""
import numpy as np
import pytest

import preprocess_oracle as po
from helpers import digest, load_golden, strided_sample

PIL = pytest.importorskip('PIL')
from PIL import Image  # noqa: E402


def _img(h, w, seed):
    g = np.random.Generator(np.random.PCG64(seed))
    base = g.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
    if seed % 2:        # smooth images exercise the rounding of long windows, noise exercises clipping
        yy, xx = np.mgrid[0:h, 0:w]
        base = np.stack([(yy * 3 + xx) % 256, (xx * 2) % 256, (yy + 2 * xx) % 256], axis=-1).astype(np.uint8)
    return base


SIZES = [((480, 640), (224, 298)), ((640, 480), (298, 224)), ((100, 75), (298, 224)), ((333, 500), (480, 720)),
         ((31, 47), (224, 224)), ((224, 224), (224, 300)), ((500, 224), (224, 224)), ((1080, 1920), (224, 398)),
         ((5, 3), (7, 2)), ((224, 224), (112, 112))]


@pytest.mark.parametrize('k', range(len(SIZES)))
def test_resize_bit_exact_vs_pillow(k):
    (h, w), (oh, ow) = SIZES[k]
    img = _img(h, w, k)
    want = np.asarray(Image.fromarray(img).resize((ow, oh), Image.BICUBIC))
    got = po.pil_resize_bicubic(img, oh, ow)
    assert got.shape == want.shape
    assert np.array_equal(got, want)


def test_size_rules_vs_torchvision():
    tv = pytest.importorskip('torchvision')
    from torchvision.transforms import Resize, CenterCrop
    for (h, w) in [(480, 640), (640, 480), (224, 224), (225, 1000), (37, 41), (1000, 225), (300, 224)]:
        for size in (224, 160, 480):
            pil = Image.fromarray(_img(h, w, 0))
            r = Resize(size, interpolation=Image.BICUBIC)(pil)
            assert (r.size[1], r.size[0]) == po.resize_shorter_edge(h, w, size)
            rh, rw = r.size[1], r.size[0]
            top, left = po.center_crop_box(rh, rw, size)
            c = np.asarray(CenterCrop(size)(r))
            assert np.array_equal(c, np.asarray(r)[top:top + size, left:left + size])


@pytest.mark.parametrize('param', [{}, {'test_crop_size': 160}, {'test_crop_size': 480, 'test_respect_ratio_max': 640},
                                   {'test_crop_size': 420, 'test_respect_ratio_max': 560}])
@pytest.mark.parametrize('hw', [(480, 640), (612, 408), (97, 301), (420, 420), (480, 480)])
def test_full_transform_vs_torchvision_pipeline(param, hw):
    """The reference's transform re-assembled from its parts (inference.py:111-132)."""
    pytest.importorskip('torchvision')
    from torchvision.transforms import Compose, Resize, CenterCrop, ToTensor, Normalize
    import torchvision.transforms.functional as F
    img = _img(hw[0], hw[1], hw[0] % 7)
    crop = param.get('test_crop_size', 224)
    if 'test_respect_ratio_max' in param:
        oh, ow = po.minmax_size(hw[0], hw[1], crop, param['test_respect_ratio_max'])
        first = [lambda im: F.resize(im, (oh, ow), interpolation=Image.BICUBIC)]
    else:
        first = [Resize(crop, interpolation=Image.BICUBIC), CenterCrop(crop), lambda im: im.convert('RGB')]
    t = Compose(first + [ToTensor(), Normalize(po.CLIP_MEAN, po.CLIP_STD)])
    want = t(Image.fromarray(img)).numpy()
    got = po.transform(img, param)
    assert got.shape == want.shape and got.dtype == np.float32
    assert np.array_equal(got, want)


@pytest.mark.parametrize('param', [{}, {'test_crop_size': 480, 'test_respect_ratio_max': 640}])
def test_equals_reference_get_image_transform(param):
    """Bit for bit against what the reference's own get_image_transform / MinMaxResizeForTest returned on these images
    (stored by oracle/make_reference_units.py: shape, sha256 of the planes and a strided sample)."""
    g = load_golden('reference_transform')
    cases = [(k, c) for k, c in enumerate(g['meta']['transform']) if c['param'] == param]
    assert len(cases) == 5
    for k, c in cases:
        got = po.transform(_img(c['hw'][0], c['hw'][1], c['img_seed']), param)
        assert list(got.shape) == c['shape']
        assert np.array_equal(strided_sample(got), g['transform_%d_sample' % k])
        assert digest(got) == c['sha256']
        if 'test_respect_ratio_max' in param:
            assert list(po.minmax_size(c['hw'][0], c['hw'][1], param['test_crop_size'],
                                       param['test_respect_ratio_max'])) == c['minmax_size']
