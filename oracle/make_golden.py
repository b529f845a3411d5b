"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.npz by running the UNMODIFIED reference
(/root/reference, imported through oracle/ref_shim.py) on seeded synthetic checkpoints.

Run in the build container only:  python oracle/make_golden.py [case ...]

The reference ships no golden vectors of its own (SURVEY.md section 4); these fixtures pin
oracle/git_oracle.py (tests/test_oracle_golden.py) and, through it and directly, the CUDA engine.
Per case we store: the config, `predictions`, `logprobs`, a strided sample of the image features
`CaptioningModel.forward_one` hands to the decoder, and for every `decoding_step` call the raw
last-position logits at 256 (64 or 32 for the big batches) fixed vocabulary columns plus the top-4 values / indices per row;
beam cases also keep the search trajectory (newest token and source row of every row at every step).
The reference's source is not modified: `decoding_step` and `image_encoder.forward` are observed by
wrapping the bound methods on the instance.
"""
import json
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

import ref_shim  # noqa: E402
from generativeimage2text_b200.synthetic import synthetic_state_dict, synthetic_images  # noqa: E402

GOLDEN_DIR = os.path.join(os.path.dirname(HERE), 'tests', 'golden')
LARGE = {'visual_feature_size': 1024, 'image_encoder_type': 'CLIPViT_L_14'}

CASES = {
    # name: param, variant, batch, frames, search, max_steps, prefix
    'base_greedy_init': dict(param={}, variant='init', batch=2, frames=0, search='greedy', max_steps=40),
    'base_greedy': dict(param={}, variant='perturbed', batch=2, frames=0, search='greedy', max_steps=40),
    'base_beam': dict(param={}, variant='init', batch=2, frames=0, search='beam', max_steps=40),
    'base_prefix': dict(param={}, variant='perturbed', batch=1, frames=1, search='greedy', max_steps=20,
                        prefix=[101, 2054, 2003, 2023]),
    'vatex_greedy': dict(param={'num_image_with_embedding': 6}, variant='perturbed', batch=1, frames=6,
                         search='greedy', max_steps=16),
    'large_greedy': dict(param=LARGE, variant='perturbed', batch=1, frames=0, search='greedy', max_steps=12),
    'large_beam': dict(param=LARGE, variant='init', batch=1, frames=0, search='beam', max_steps=12),
    # MinMaxResizeForTest-style input: a 160-crop model (10x10 grid embedding) fed 160x208 pixels (10x13 grid) ->
    # run-time positional-embedding interpolation (reference layers/CLIP/model.py:245-251)
    'base_ratio_greedy': dict(param={'test_crop_size': 160, 'test_respect_ratio_max': 224}, variant='perturbed', batch=2,
                              frames=0, search='greedy', max_steps=12, image_hw=[160, 208]),
    # the shipped GIT_BASE_VQAv2 / TEXTVQA geometry (aux_data/models/GIT_BASE_VQAv2/parameter.yaml): 480-crop model
    # (30x30 grid embedding), a 480x640 input (30x40 grid = 1201 image tokens) and a question prefix
    'base_vqa_ratio_greedy': dict(param={'test_crop_size': 480, 'test_respect_ratio_max': 640}, variant='perturbed', batch=1,
                                  frames=1, search='greedy', max_steps=10, image_hw=[480, 640], prefix=[101, 2054, 2003, 2023]),
    # square non-default crop: the embedding is built for the 10x10 grid, no run-time interpolation
    'base_crop160_greedy': dict(param={'test_crop_size': 160}, variant='perturbed', batch=2, frames=1, search='greedy',
                                max_steps=12, image_hw=[160, 160]),
    # ---- round 2: the benchmarked configurations themselves (BASELINE.json configs 2-4; bench.py's checkpoints and pixels)
    'base_greedy_b64': dict(param={}, variant='init', batch=64, frames=0, search='greedy', max_steps=40, n_cols=64),
    # (every other of the 64 sampled columns: 128 rows x 39 steps of logits keep the file under 1 MB)
    'large_beam_b32': dict(param=LARGE, variant='init', batch=32, frames=0, search='beam', max_steps=40, n_cols=64,
                           col_stride=2),
    'vatex_greedy_b16': dict(param={'num_image_with_embedding': 6}, variant='init', batch=16, frames=6, search='greedy',
                             max_steps=40, n_cols=64),
    # ---- decisive-margin checkpoints (SURVEY.md section 7 hard part 1b): free-running token identity is asserted on these.
    # (weight seed, image seed) come out of tools/decisive_sweep.py; `min_margin` is recorded in the file.
    'base_decisive': dict(param={}, variant='decisive', batch=4, frames=0, search='greedy', max_steps=20, img_seed=5030),
}


def vocab_sample(n=256):
    g = np.random.Generator(np.random.PCG64(777))
    return np.sort(g.choice(30522, size=n, replace=False)).astype(np.int64)


def beam_idx_from_histories(prev_ids, ids, beam):
    """The reference re-orders `input_ids[beam_idx]` inside its search loop (layers/decoder.py:1231) without exposing
    beam_idx; recover, per row, a source row of the same image whose previous history equals this row's history minus its
    newest token (rows with identical histories have identical text K/V, so any of them is the same re-ordering)."""
    rows = ids.shape[0]
    out = np.zeros(rows, dtype=np.int32)
    for r in range(rows):
        b0 = (r // beam) * beam
        want = ids[r, :-1]
        src = [k for k in range(b0, b0 + beam) if np.array_equal(prev_ids[k], want)]
        if not src:   # finished image: the reference pads with global row 0 (layers/decoder.py:1189)
            src = [k for k in range(rows) if np.array_equal(prev_ids[k], want)]
        assert src, 'no source row for row %d' % r
        out[r] = src[0]
    return out


def run_case(name, cfg, seed=0, img_seed=1234):
    seed = cfg.get('seed', seed)
    img_seed = cfg.get('img_seed', img_seed)
    sd = synthetic_state_dict(cfg['param'], seed, cfg['variant'])
    model = ref_shim.load_reference_model(cfg['param'], cfg['search'], cfg['max_steps'], state_dict=sd)
    image = synthetic_images(cfg['batch'], cfg['frames'], img_seed, cfg.get('image_hw', 224))
    batch = {'image': image}
    if 'prefix' in cfg:
        batch['prefix'] = torch.tensor([cfg['prefix']], dtype=torch.long)
    cols = torch.from_numpy(vocab_sample(cfg.get('n_cols', 256))[::cfg.get('col_stride', 1)].copy())
    steps, inputs = [], []
    orig = model.decoding_step

    def spy(*a, **kw):
        z = orig(*a, **kw)
        top = z.topk(4, dim=1)
        steps.append((z[:, cols].clone(), top.values.clone(), top.indices.clone()))
        inputs.append(a[3].clone())          # partial_captions of this call [rows, cur_len]
        return z
    model.decoding_step = spy
    t0 = time.time()
    with torch.no_grad():
        out = model(batch)
        # image features as the decoder sees them (reference layers/decoder.py:846-857)
        if isinstance(image, (list, tuple)):
            fs = [model.image_encoder(im) for im in image]
            if model.num_image_with_embedding:
                fs = [f + e for f, e in zip(fs, model.img_temperal_embedding)]
            vf = torch.cat(fs, dim=1)
        else:
            vf = model.image_encoder(image)
        vproj = model.textual.visual_projection(vf)
    dt = time.time() - t0
    extra = {}
    if cfg['search'] == 'beam':
        # the trajectory of the reference's search: per step the newest input token of every row and the re-ordering that
        # produced its history (drives the engine's raw decode-step API in tests/test_gpu_parity.py)
        ids = [x.numpy() for x in inputs]
        extra['step_tokens'] = np.stack([x[:, -1] for x in ids])
        bidx = [np.arange(ids[0].shape[0], dtype=np.int32)]
        for prev, cur in zip(ids[:-1], ids[1:]):
            bidx.append(beam_idx_from_histories(prev, cur, 4))
        extra['step_beam_idx'] = np.stack(bidx)
    if cfg['variant'] == 'decisive':
        # smallest top-1 / top-2 gap of the reference's own free-running decisions (after its no-repeat scatter; rows that
        # already ended are EOS-forced and excluded)
        pred = out['predictions']
        mins = []
        for i, (_, tv, ti) in enumerate(steps):
            for r in range(pred.shape[0]):
                if i > 0 and pred[r, i].item() == 102:
                    continue
                vals = [v for v, t in zip(tv[r].tolist(), ti[r].tolist()) if not (i > 0 and t == pred[r, i].item())]
                mins.append(vals[0] - vals[1])
        extra['min_margin'] = np.array(min(mins), dtype=np.float64)
    meta = dict(cfg)
    meta.update(seed=seed, img_seed=img_seed, reference_commit='faae4fb9', torch=torch.__version__,
                generator='oracle/make_golden.py', seconds=round(dt, 2))
    np.savez_compressed(
        os.path.join(GOLDEN_DIR, name + '.npz'),
        meta=np.array(json.dumps(meta)),
        predictions=out['predictions'].numpy(),
        logprobs=out['logprobs'].numpy(),
        vocab_cols=cols.numpy(),
        step_logits=torch.stack([s[0] for s in steps]).numpy(),
        step_top2_val=torch.stack([s[1][:, :2] for s in steps]).numpy(),
        step_top2_idx=torch.stack([s[2][:, :2] for s in steps]).numpy(),
        step_top4_val=torch.stack([s[1] for s in steps]).numpy(),
        step_top4_idx=torch.stack([s[2] for s in steps]).numpy(),
        feats_sample=vf[:, ::17, ::29].numpy(),
        vproj_sample=vproj[:, ::17, ::29].numpy(),
        feats_absmean=np.array(vf.abs().mean().item(), dtype=np.float64),
        **extra
    )
    print('%-18s %5.1fs steps=%d pred=%s lp=%s' % (
        name, dt, len(steps), tuple(out['predictions'].shape),
        np.round(out['logprobs'].flatten().numpy(), 4).tolist()))


if __name__ == '__main__':
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    torch.set_num_threads(os.cpu_count())
    names = sys.argv[1:] or list(CASES)
    for n in names:
        run_case(n, CASES[n])
