"""CPU: oracle/git_oracle.py and the model's state-dict layout against what the reference's own modules returned on the
same inputs (stored by oracle/make_reference_units.py)."""
import pytest
import torch

import git_oracle
from generativeimage2text_b200.model import get_git_model
from generativeimage2text_b200.synthetic import state_spec, synthetic_state_dict, synthetic_images
from helpers import load_golden


class Tok:
    cls_token_id, sep_token_id = 101, 102


def test_state_dict_layout_matches_reference():
    for ref in load_golden('reference_model')['meta']['layout']:
        param = ref['param']
        spec = state_spec(param)
        assert [[k, list(shp)] for k, shp, _ in spec] == ref['keys']
        # the same tensors share storage (the LM head is the word embedding)
        groups = {}
        for k, v in get_git_model(Tok(), param).state_dict().items():
            groups.setdefault(v.data_ptr(), []).append(k)
        assert [g for g in groups.values() if len(g) > 1] == ref['tied']


@pytest.mark.parametrize('search', ['greedy', 'beam'])
def test_oracle_equals_reference_fresh_seed(search):
    """A seed/image set that is NOT in tests/golden."""
    g = load_golden('reference_model')
    f = g['meta']['fresh']
    sd = synthetic_state_dict({}, seed=f['weight_seed'], variant=f['variant'])
    img = synthetic_images(1, 0, seed=f['img_seed'])
    rp = torch.from_numpy(g['fresh_%s_predictions' % search])
    rl = torch.from_numpy(g['fresh_%s_logprobs' % search])
    for cached in (True, False):
        o = git_oracle.generate(sd, {}, {'image': img}, search, f['max_steps'], cached=cached)
        assert torch.equal(rp, o['predictions'])
        assert torch.allclose(rl, o['logprobs'], atol=1e-3)


# ---- the remaining decoders (SURVEY.md 8f-4): vocabulary trie, sampling ------------------------------------------------
def _toy_step(vocab=64, seed=3):
    """Deterministic stand-in for `decoding_step`: logits depend on the row's last token and on the caption length."""
    g = torch.Generator().manual_seed(seed)
    table = torch.randn(vocab, vocab, generator=g) * 2.0
    drift = torch.randn(64, vocab, generator=g) * 0.5

    def step(partial):
        return table[partial[:, -1]] + drift[partial.shape[1]]
    return step


def _toy_trie_sequences(eos):
    return [[5, 9, 11, eos], [5, 9, 12, 13, eos], [5, 20, eos], [7, 9, eos], [7, 30, 31, 32, eos], [40, eos]]


def test_trie_search_equals_reference():
    """oracle/git_oracle.trie_search against the reference's TrieAutoRegressiveBeamSearch (trie_decoder.py:27-218) at batch 1,
    the case that decoder supports (with more rows its single cursor follows row 0 only and `TokenTrie.move` asserts as
    soon as row 0 has ended while another row has not): verbatim mode and the per-row mode the engine implements."""
    B = 1
    from generativeimage2text_b200.model import TokenTrie
    g = load_golden('reference_model')
    eos = 2
    seqs = _toy_trie_sequences(eos)
    start = torch.tensor([[1]] * B)
    assert g['meta']['trie_seeds'] == 4
    for seed in range(4):
        step = _toy_step(seed=seed)
        rp, rl = torch.from_numpy(g['trie_%d_predictions' % seed]), torch.from_numpy(g['trie_%d_logprobs' % seed])
        csr = TokenTrie.construct(seqs).to_csr()
        op, ol = git_oracle.trie_search(start, step, csr, max_steps=12, eos=eos, per_row=False)
        assert torch.equal(rp, op) and torch.allclose(rl, ol, atol=1e-5)
        pp, pl = git_oracle.trie_search(start, step, csr, max_steps=12, eos=eos, per_row=True)
        assert torch.equal(rp, pp) and torch.allclose(rl, pl, atol=1e-5)
        assert rp[0, 1:].tolist() in seqs                   # the constraint binds: the caption is one of the trie's sequences


def test_trie_search_per_row_is_batch_of_batch1_calls():
    from generativeimage2text_b200.model import TokenTrie
    eos = 2
    csr = TokenTrie.construct(_toy_trie_sequences(eos)).to_csr()
    g = torch.Generator().manual_seed(11)
    table = torch.randn(3, 64, 64, generator=g) * 2.0          # a different "image" per row

    def step_rows(rows):
        def step(partial):
            return torch.stack([table[r][partial[i, -1]] + 0.1 * partial.shape[1] for i, r in enumerate(rows)])
        return step
    start = torch.tensor([[1]] * 3)
    bp, bl = git_oracle.trie_search(start, step_rows([0, 1, 2]), csr, max_steps=10, eos=eos)
    for r in range(3):
        p1, l1 = git_oracle.trie_search(start[:1], step_rows([r]), csr, max_steps=10, eos=eos)
        n = p1.shape[1]
        assert torch.equal(bp[r, :n], p1[0]) and bool((bp[r, n:] == eos).all())
        assert torch.allclose(bl[r], l1[0], atol=1e-5)


@pytest.mark.parametrize('temperature', [1.0, 0.7])
def test_sample_search_equals_reference_with_the_same_draws(temperature):
    """The do_sample branches of the reference's AutoRegressiveBeamSearch.search (layers/decoder.py:260-276, 364-375) with
    torch.multinomial replaced by the inverse-CDF draw the engine makes, fed the same uniforms."""
    g = load_golden('reference_model')
    eos, B, steps = 2, 4, 14
    start = torch.tensor([[1]] * B)
    u = torch.rand((steps, B), generator=torch.Generator().manual_seed(5))
    assert g['meta']['sample_seeds'] == 3
    for seed in range(3):
        step = _toy_step(seed=seed)
        rp = torch.from_numpy(g['sample_%g_%d_predictions' % (temperature, seed)])
        rl = torch.from_numpy(g['sample_%g_%d_logprobs' % (temperature, seed)])
        op, ol = git_oracle.sample_search(start, step, u, temperature=temperature, max_steps=steps, eos=eos)
        assert torch.equal(rp, op)
        assert torch.allclose(rl, ol, atol=1e-5)
