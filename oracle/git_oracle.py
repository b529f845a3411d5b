"""TEST INFRASTRUCTURE ONLY -- CPU restatement (fp32, plain torch ops) of the reference's GIT
captioning hot path.  It is the *checker* for the CUDA engine and the `cpu_baseline` leg of
bench.py; the product package never imports it (the product fails loudly without its CUDA library).

Parity status: the reference ships no tests or golden vectors (SURVEY.md section 4), so this
restatement is pinned against outputs of the reference's own modules:
  * tests/test_oracle_vs_reference.py compares it with what the reference returned on the same seeded weights/pixels
    (tests/golden/reference_model.npz, recorded by oracle/make_reference_units.py);
  * tests/golden/*.npz were produced by the *unmodified reference* (oracle/make_golden.py) and are
    checked against this file on every machine (tests/test_oracle_golden.py).

Every function cites the reference file:line it follows (paths relative to
/root/reference/generativeimage2text/).  Two execution modes of the decoder:
  * `CachedDecoder`   -- KV-cached single-row steps (results-equivalent, SURVEY.md Appendix A
                         "KV-cache equivalence"); used for checking, it is what the engine implements.
  * `as_shipped_step` -- recomputes the whole [image || text] sequence every step exactly like the
                         shipped reference (SURVEY.md section 0 item 1); used for the CPU baseline timing.
"""
import math

import torch
import torch.nn.functional as F

EOS = 102
CLS = 101

ENCODER_CFG = {
    'CLIPViT_B_16': dict(patch=16, width=768, layers=12, heads=12),
    'CLIPViT_L_14': dict(patch=14, width=1024, layers=24, heads=16),
}
DEC_LAYERS = 6
DEC_HEADS = 12


def _ln(x, sd, prefix, eps):
    return F.layer_norm(x, (x.shape[-1],), sd[prefix + '.weight'], sd[prefix + '.bias'], eps)


# ----------------------------------------------------------------------------------------------
# hot path A: CLIP ViT image encoder
# ----------------------------------------------------------------------------------------------
def encode_image(sd, param, img, taps=None):
    """VisualTransformer.forward with output_grid=grid_after_ln=True (layers/CLIP/model.py:240-268).

    img fp32 [B,3,H,W] -> [B, L, d].  ResidualAttentionBlock: layers/CLIP/model.py:189-202;
    QuickGELU :171-173; LayerNorm eps 1e-5 (nn.LayerNorm default, :161-168).
    """
    cfg = ENCODER_CFG[(param or {}).get('image_encoder_type', 'CLIPViT_B_16')]
    p, d, nl, nh = cfg['patch'], cfg['width'], cfg['layers'], cfg['heads']
    pre = 'image_encoder.'
    B = img.shape[0]
    x = F.conv2d(img, sd[pre + 'conv1.weight'], None, stride=p)                # :242
    pos = sd[pre + 'positional_embedding']
    g0 = int(round(math.sqrt(pos.shape[0] - 1)))                                # expected_dim :243
    if x.shape[2] != g0 or x.shape[3] != g0:                                    # :245-251 run-time re-sampling
        grid = pos[1:, :].reshape(g0, g0, d).permute(2, 0, 1).unsqueeze(0)
        grid = F.interpolate(grid, size=(x.shape[2], x.shape[3]), mode='bicubic')
        pos = torch.cat((pos[0:1, :], grid.squeeze(0).permute(1, 2, 0).reshape(-1, d)), dim=0)
    x = x.reshape(B, d, -1).permute(0, 2, 1)                                  # :252-253
    cls = sd[pre + 'class_embedding'].expand(B, 1, d)
    x = torch.cat([cls, x], dim=1) + pos                                      # :254-255
    x = _ln(x, sd, pre + 'ln_pre', 1e-5)                                      # :257
    if taps is not None:
        taps['ln_pre'] = x
    L = x.shape[1]
    hd = d // nh
    for i in range(nl):
        b = pre + 'transformer.resblocks.%d.' % i
        h = _ln(x, sd, b + 'ln_1', 1e-5)
        qkv = F.linear(h, sd[b + 'attn.in_proj_weight'], sd[b + 'attn.in_proj_bias'])
        q, k, v = qkv.split(d, dim=-1)
        q = q.reshape(B, L, nh, hd).transpose(1, 2)
        k = k.reshape(B, L, nh, hd).transpose(1, 2)
        v = v.reshape(B, L, nh, hd).transpose(1, 2)
        att = torch.softmax((q @ k.transpose(-1, -2)) / math.sqrt(hd), dim=-1)  # SDPA, no mask
        ctx = (att @ v).transpose(1, 2).reshape(B, L, d)
        x = x + F.linear(ctx, sd[b + 'attn.out_proj.weight'], sd[b + 'attn.out_proj.bias'])  # :200
        h = _ln(x, sd, b + 'ln_2', 1e-5)
        u = F.linear(h, sd[b + 'mlp.c_fc.weight'], sd[b + 'mlp.c_fc.bias'])
        u = u * torch.sigmoid(1.702 * u)                                      # QuickGELU :171-173
        x = x + F.linear(u, sd[b + 'mlp.c_proj.weight'], sd[b + 'mlp.c_proj.bias'])          # :201
        if taps is not None and i == 0:
            taps['block0'] = x
    return _ln(x, sd, pre + 'ln_post', 1e-5)                                  # :263-268 (all tokens)


def visual_features(sd, param, image):
    """CaptioningModel.forward_one image branch (layers/decoder.py:846-857): per-frame encoder,
    `+ img_temperal_embedding[i]` (zip truncates), concat on the token axis."""
    if isinstance(image, (list, tuple)):
        feats = [encode_image(sd, param, im) for im in image]
        n_emb = (param or {}).get('num_image_with_embedding') or 0
        if n_emb:
            feats = [f + sd['img_temperal_embedding.%d' % i] for i, f in zip(range(n_emb), feats)]
        return torch.cat(feats, dim=1)
    return encode_image(sd, param, image)


def project_visual(sd, feats):
    """visual_projection = Linear(dv->768) + LayerNorm(eps 1e-5) (layers/decoder.py:30-36, 535)."""
    t = 'textual.visual_projection.'
    return _ln(F.linear(feats, sd[t + '0.weight'], sd[t + '0.bias']), sd, t + '1', 1e-5)


def embed_tokens(sd, tokens, first_pos=0):
    """WordAndPositionalEmbedding (layers/decoder.py:65-78): LN(words[tok] + positions[i], eps 1e-8)."""
    t = 'textual.embedding.'
    pos = torch.arange(first_pos, first_pos + tokens.shape[1])
    e = sd[t + 'words.weight'][tokens] + sd[t + 'positions.weight'][pos]
    return _ln(e, sd, t + 'layer_norm', 1e-8)


def _gelu_erf(x):
    """layers/bert/activations.py:16-23."""
    return x * 0.5 * (1.0 + torch.erf(x / math.sqrt(2.0)))


def _bert_layer(sd, j, x_q, k_all, v_all, mask):
    """One post-norm BertLayer (layers/bert/modeling_bert.py:124-152, 171-178, 228-231, 243-250)
    for query rows x_q against already-projected keys/values. mask broadcastable to [B,H,Sq,Sk]."""
    b = 'textual.transformer.encoder.layer.%d.' % j
    B, Sq, D = x_q.shape
    H, hd = DEC_HEADS, D // DEC_HEADS
    q = F.linear(x_q, sd[b + 'attention.self.query.weight'], sd[b + 'attention.self.query.bias'])
    q = q.reshape(B, Sq, H, hd).transpose(1, 2)
    k = k_all.reshape(B, -1, H, hd).transpose(1, 2)
    v = v_all.reshape(B, -1, H, hd).transpose(1, 2)
    s = (q / math.sqrt(hd)) @ k.transpose(-1, -2)                 # qk2attn :41-47 (Q scaled first)
    if mask is not None:
        s = s + mask
    ctx = (s.softmax(dim=-1) @ v).transpose(1, 2).reshape(B, Sq, D)
    a = F.linear(ctx, sd[b + 'attention.output.dense.weight'], sd[b + 'attention.output.dense.bias'])
    a = _ln(a + x_q, sd, b + 'attention.output.LayerNorm', 1e-12)
    u = _gelu_erf(F.linear(a, sd[b + 'intermediate.dense.weight'], sd[b + 'intermediate.dense.bias']))
    y = F.linear(u, sd[b + 'output.dense.weight'], sd[b + 'output.dense.bias'])
    return _ln(y + a, sd, b + 'output.LayerNorm', 1e-12)


def _kv(sd, j, x):
    b = 'textual.transformer.encoder.layer.%d.attention.self.' % j
    return (F.linear(x, sd[b + 'key.weight'], sd[b + 'key.bias']),
            F.linear(x, sd[b + 'value.weight'], sd[b + 'value.bias']))


def lm_head(sd, y):
    """Tied output layer (layers/decoder.py:503-505, 587)."""
    return F.linear(y, sd['textual.embedding.words.weight'], sd['textual.output.bias'])


# ----------------------------------------------------------------------------------------------
# hot path B, as shipped: full recompute every step
# ----------------------------------------------------------------------------------------------
def as_shipped_step(sd, vis_feats, partial_captions):
    """CaptioningModel.decoding_step with prev_encoded_layers=None (layers/decoder.py:1013-1054):
    beam-expand features (:1019-1025), visual_projection on all image tokens every step (:535),
    embed all text tokens, [image || text] through 6 layers with the block mask of
    BertEncoderAsDecoder.forward (:114-137), LM head on all text rows, keep the last (:1054)."""
    R, t = partial_captions.shape
    B, M, _ = vis_feats.shape
    beam = R // B
    if beam > 1:
        vis_feats = vis_feats.unsqueeze(1).repeat(1, beam, 1, 1).view(R, M, -1)
    v = project_visual(sd, vis_feats)
    e = embed_tokens(sd, partial_captions)
    x = torch.cat([v, e], dim=1)
    S = M + t
    mask = torch.zeros(S, S)
    mask[:M, M:] = float('-inf')                                                   # :119-120
    mask[M:, M:] = torch.triu(torch.full((t, t), float('-inf')), diagonal=1)      # :602-610
    mask = mask[None, None]
    for j in range(DEC_LAYERS):
        k, vv = _kv(sd, j, x)
        x = _bert_layer(sd, j, x, k, vv, mask)
    logits = lm_head(sd, x[:, M:])
    return logits[:, -1, :].float()


# ----------------------------------------------------------------------------------------------
# hot path B, KV-cached (what the engine implements)
# ----------------------------------------------------------------------------------------------
class CachedDecoder(object):
    """Image rows never attend to text (layers/decoder.py:119-120) so their K/V are computed once
    (`prefill`); each step computes only the newest text row per sequence (`step`).  Under beam
    search the text K/V follow `input_ids[beam_idx]` (layers/decoder.py:1231) -> `reorder`."""

    def __init__(self, sd, vis_feats, beam=1, taps=None):
        self.sd = sd
        self.beam = beam
        v = project_visual(sd, vis_feats)                      # [B, M, D]
        if taps is not None:
            taps['visual_projection'] = v
        self.B, self.M, self.D = v.shape
        self.img_k, self.img_v = [], []
        x = v
        for j in range(DEC_LAYERS):
            k, vv = _kv(sd, j, x)
            self.img_k.append(k)
            self.img_v.append(vv)
            if j + 1 < DEC_LAYERS:                             # image rows of the last layer are unused
                x = _bert_layer(sd, j, x, k, vv, None)
                if taps is not None:
                    taps['prefill_layer%d' % j] = x
        R = self.B * beam
        self.txt_k = [torch.zeros(R, 0, self.D) for _ in range(DEC_LAYERS)]
        self.txt_v = [torch.zeros(R, 0, self.D) for _ in range(DEC_LAYERS)]
        self.n_text = 0

    def _expand(self, t):
        if self.beam == 1:
            return t
        return t.unsqueeze(1).expand(-1, self.beam, -1, -1).reshape(self.B * self.beam, *t.shape[1:])

    def feed(self, tokens):
        """Append `tokens` [R, n] (n >= 1) at positions n_text.. and return last-row logits [R, V]."""
        sd = self.sd
        n = tokens.shape[1]
        x = embed_tokens(sd, tokens, first_pos=self.n_text)
        mask = None
        if n > 1:   # prefix tokens fed at once: causal among themselves, all see image + earlier text
            mask = torch.zeros(n, self.M + self.n_text + n)
            mask[:, self.M + self.n_text:] = torch.triu(torch.full((n, n), float('-inf')), diagonal=1)
            mask = mask[None, None]
        for j in range(DEC_LAYERS):
            k, v = _kv(sd, j, x)
            self.txt_k[j] = torch.cat([self.txt_k[j], k], dim=1)
            self.txt_v[j] = torch.cat([self.txt_v[j], v], dim=1)
            k_all = torch.cat([self._expand(self.img_k[j]), self.txt_k[j]], dim=1)
            v_all = torch.cat([self._expand(self.img_v[j]), self.txt_v[j]], dim=1)
            x = _bert_layer(sd, j, x, k_all, v_all, mask)
        self.n_text += n
        return lm_head(sd, x[:, -1]).float()

    def reorder(self, beam_idx):
        self.txt_k = [k[beam_idx] for k in self.txt_k]
        self.txt_v = [v[beam_idx] for v in self.txt_v]


# ----------------------------------------------------------------------------------------------
# search loops
# ----------------------------------------------------------------------------------------------
def greedy_search(start, step, max_steps=40, eos=EOS, trace=None):
    """AutoRegressiveBeamSearch.search with beam_size=1, per_node_beam_size=1,
    fix_missing_prefix=True (layers/decoder.py:224-440; the reference's greedy, model.py:27-33).

    `step(partial_captions [B,t]) -> logits [B,V]`.  Returns (predictions incl. the start tokens,
    logprobs / num_valid).  `trace`, if a list, receives (logits_after_masking, top2 margin) per step.
    """
    B, P = start.shape
    logits = step(start)                                                        # :258
    ls = F.log_softmax(logits, dim=1)                                           # :265
    lp, tok = ls.max(dim=1)                                                     # topk(1) :271
    if trace is not None:
        trace.append(logits.clone())
    if bool((tok == eos).all()):                                                # :279-291
        return tok[:, None], lp[:, None]
    pred = torch.cat([start, tok[:, None]], dim=1)                              # :298
    while pred.shape[1] < max_steps:                                            # :313
        last = pred[:, -1]
        if bool((last == eos).all()):                                           # :319
            break
        z = step(pred)
        z = z.scatter(1, last[:, None], -10000.0)                               # no-repeat :330
        done = last == eos
        if bool(done.any()):                                                    # EOS forcing :347-351
            forced = torch.full_like(z, float('-inf'))
            forced[:, eos] = 0.0
            z = torch.where(done[:, None], forced, z)
        if trace is not None:
            trace.append(z.clone())
        ls = F.log_softmax(z, dim=1)                                            # :358
        slp, tok = ls.max(dim=1)                                                # :366
        lp = lp + slp                                                           # :386, :408-416 (beam 1)
        pred = torch.cat([pred, tok[:, None]], dim=1)
    num_valid = (pred != eos).sum(dim=-1)                                       # :433-438
    num_valid = num_valid + ((pred == eos).sum(dim=-1) > 0).long()
    num_valid = (num_valid - P).clip(min=1)
    return pred, lp / num_valid


def trie_csr_children(csr, node):
    """(tokens, child nodes) of `node` in the CSR form the engine takes (include/gitb200.h gitb200_set_trie)."""
    begin, tok, child = csr
    return tok[begin[node]:begin[node + 1]], child[begin[node]:begin[node + 1]]


def trie_search(start, step, csr, max_steps=40, eos=EOS, per_row=True):
    """TrieAutoRegressiveBeamSearch.search (trie_decoder.py:44-218; beam_size is asserted 1, :38): greedy decoding in which
    the log-probs of the tokens the trie allows next are raised by (max logit - min logit + 1) before the top-1.

    per_row=False is the reference verbatim: ONE cursor, only row 0 is raised (:61-62, :141-142) and moved (:70, :153), max /
    min over the whole [B, V] matrix.  per_row=True is what the engine implements: every row owns a cursor and is treated as a
    batch-1 call (max / min over its own row; a row that already ended with EOS is EOS-forced and keeps its cursor).  For
    B = 1 both are the same thing."""
    B, P = start.shape
    cur = [0] * B

    def raise_allowed(ls, z, rows):
        for r in rows:
            toks, _ = trie_csr_children(csr, cur[r])
            if len(toks):
                zz = z[r] if per_row else z
                ls[r, torch.tensor(toks, dtype=torch.long)] += zz.max() - zz.min() + 1          # :62 / :142

    def move(tok, rows):
        for r in rows:
            toks, kids = trie_csr_children(csr, cur[r])
            t = int(tok[r])
            assert t in toks, 'token %d is not allowed at node %d' % (t, cur[r])      # TokenTrie.move :257
            cur[r] = kids[toks.index(t)]

    rows0 = list(range(B)) if per_row else [0]
    logits = step(start)                                                        # :58
    ls = F.log_softmax(logits, dim=1)                                           # :59
    raise_allowed(ls, logits, rows0)
    lp, tok = ls.max(dim=1)                                                     # topk(1) :67
    move(tok, rows0)
    if bool((tok == eos).all()):                                                # :72-79
        return tok[:, None], lp[:, None]
    pred = torch.cat([start, tok[:, None]], dim=1)                              # :86
    while pred.shape[1] < max_steps:                                            # :101
        last = pred[:, -1]
        if bool((last == eos).all()):                                           # :107
            break
        z = step(pred)
        z = z.scatter(1, last[:, None], -10000.0)                               # :122
        done = last == eos
        if bool(done.any()):                                                    # :134-138
            forced = torch.full_like(z, float('-inf'))
            forced[:, eos] = 0.0
            z = torch.where(done[:, None], forced, z)
        ls = F.log_softmax(z, dim=1)                                            # :140
        live = [r for r in rows0 if not bool(done[r])] if per_row else rows0
        raise_allowed(ls, z, live)
        slp, tok = ls.max(dim=1)                                                # :150
        move(tok, live)
        lp = lp + slp                                                           # :163, :190-199 (beam 1)
        pred = torch.cat([pred, tok[:, None]], dim=1)
    num_valid = (pred != eos).sum(dim=-1)                                       # :206-211
    num_valid = num_valid + ((pred == eos).sum(dim=-1) > 0).long()
    num_valid = (num_valid - P).clip(min=1)
    return pred, lp / num_valid


def inverse_cdf_draw(probs, u):
    """One index per row of `probs` [B, V]: the first i with cumsum(probs)[i] > u * sum(probs) -- the draw the engine makes in
    place of torch.multinomial (whose random stream cannot be reproduced); float64 accumulation."""
    c = torch.cumsum(probs.double(), dim=1)
    target = u.double() * c[:, -1]
    idx = (c > target[:, None]).float().argmax(dim=1)
    none = ~(c > target[:, None]).any(dim=1)
    return torch.where(none, torch.full_like(idx, probs.shape[1] - 1), idx)


def sample_search(start, step, uniforms, temperature=1.0, max_steps=40, eos=EOS, draw=inverse_cdf_draw):
    """The do_sample=True branches of AutoRegressiveBeamSearch.search with beam_size = per_node_beam_size = 1
    (layers/decoder.py:224-440): the first token is drawn from softmax(logits / T) and scored with log_softmax(logits / T)
    (:259-272); later tokens are drawn from softmax(z / T) but scored with log_softmax(z) of the UN-tempered masked logits
    (:358 before :369-370).  `uniforms[t, r]` drives the draw of row r at caption length t."""
    B, P = start.shape
    logits = step(start) / temperature                                          # :258-261
    ls = F.log_softmax(logits, dim=1)                                           # :265
    tok = draw(logits.softmax(dim=1), uniforms[P])                              # :274-275
    lp = ls.gather(1, tok[:, None])[:, 0]                                       # :276
    if bool((tok == eos).all()):                                                # :279-291
        return tok[:, None], lp[:, None]
    pred = torch.cat([start, tok[:, None]], dim=1)
    while pred.shape[1] < max_steps:
        last = pred[:, -1]
        if bool((last == eos).all()):
            break
        z = step(pred)
        z = z.scatter(1, last[:, None], -10000.0)                               # :330
        done = last == eos
        if bool(done.any()):                                                    # :347-351
            forced = torch.full_like(z, float('-inf'))
            forced[:, eos] = 0.0
            z = torch.where(done[:, None], forced, z)
        ls = F.log_softmax(z, dim=1)                                            # :358
        tok = draw((z / temperature).softmax(dim=1), uniforms[pred.shape[1]])   # :369-373
        tok = torch.where(done, torch.full_like(tok, eos), tok)                 # a one-hot distribution has one outcome
        lp = lp + ls.gather(1, tok[:, None])[:, 0]                              # :374, :386
        pred = torch.cat([pred, tok[:, None]], dim=1)
    num_valid = (pred != eos).sum(dim=-1)                                       # :433-438
    num_valid = num_valid + ((pred == eos).sum(dim=-1) > 0).long()
    num_valid = (num_valid - P).clip(min=1)
    return pred, lp / num_valid


def _length_norm(length, lp):
    """BeamHypotheses._length_norm (layers/decoder.py:1310-1313)."""
    return (5 + length) ** lp / (5 + 1) ** lp


def beam_search(start, step, reorder=None, max_steps=40, beam=4, per_node=2, length_penalty=0.6,
                eos=EOS, trace=None):
    """GeneratorWithBeamSearch.search, greedy branch, num_keep_best=1 (layers/decoder.py:1083-1290)
    with BeamHypotheses (:1292-1341).

    `step(input_ids [B*beam, t]) -> logits [B*beam, V]`; `reorder(beam_idx)` is called before the
    next step when a KV cache has to follow `input_ids[beam_idx]` (:1231; the reference's own
    re-order code is commented out because it has no cache).
    Returns (decoded [B, max_steps] EOS-padded, logprobs [B,1]).
    """
    B, cur_len = start.shape
    ids = start.unsqueeze(1).expand(B, beam, cur_len).reshape(B * beam, cur_len)
    max_length = max_steps
    hyps = [dict(hyp=[], worst=1e9) for _ in range(B)]                          # n_hyp = 1

    def hyp_add(h, seq, sum_lp):                                                # :1315-1328
        score = sum_lp / _length_norm(len(seq), length_penalty)
        if len(h['hyp']) < 1 or score > h['worst']:
            h['hyp'].append((score, seq))
            if len(h['hyp']) > 1:
                srt = sorted([(s, i) for i, (s, _) in enumerate(h['hyp'])])
                del h['hyp'][srt[0][1]]
                h['worst'] = srt[1][0]
            else:
                h['worst'] = min(score, h['worst'])

    def hyp_done(h, best_sum_lp):                                               # :1330-1341
        if len(h['hyp']) < 1:
            return False
        return h['worst'] >= best_sum_lp / _length_norm(max_length - 1, length_penalty)

    beam_scores = torch.zeros(B, beam)
    beam_scores[:, 1:] = -1e9                                                   # :1118-1120
    beam_scores = beam_scores.view(-1)
    done = [False] * B
    while cur_len < max_length:                                                 # :1129
        logits = step(ids)
        V = logits.shape[-1]
        scores = F.log_softmax(logits, dim=-1) + beam_scores[:, None]           # :1169-1172
        if trace is not None:
            trace.append(logits.clone())
        nscore, nword = torch.topk(scores.view(B, beam * V), per_node * beam, dim=1,
                                   largest=True, sorted=True)                   # :1175
        nxt = []
        for b in range(B):
            done[b] = done[b] or hyp_done(hyps[b], nscore[b].max().item())      # :1187
            if done[b]:
                nxt.extend([(0.0, eos, 0)] * beam)                              # :1189 (global row 0)
                continue
            sent = []
            for idx, sc in zip(nword[b].tolist(), nscore[b].tolist()):
                bid, wid = idx // V, idx % V
                if wid == eos or cur_len + 1 == max_length:                     # :1202-1206
                    hyp_add(hyps[b], ids[b * beam + bid, :cur_len].clone(), sc)
                else:
                    sent.append((sc, wid, b * beam + bid))
                if len(sent) == beam:
                    break
            if len(sent) == 0:
                sent = [(0.0, eos, 0)] * beam
            assert len(sent) == beam
            nxt.extend(sent)
        beam_scores = torch.tensor([x[0] for x in nxt], dtype=torch.float32)
        words = torch.tensor([x[1] for x in nxt], dtype=torch.long)
        bidx = torch.tensor([x[2] for x in nxt], dtype=torch.long)
        ids = torch.cat([ids[bidx], words[:, None]], dim=-1)                    # :1231-1232
        if reorder is not None:
            reorder(bidx)
        cur_len += 1
        if all(done):
            break
    decoded = torch.full((B, max_length), eos, dtype=torch.long)                # :1283
    logprobs = torch.full((B, 1), -1e5)
    for b in range(B):
        if hyps[b]['hyp']:
            sc, seq = max(hyps[b]['hyp'], key=lambda x: x[0])
            logprobs[b, 0] = sc
            decoded[b, :len(seq)] = seq
            decoded[b, len(seq)] = eos
    return decoded, logprobs


# ----------------------------------------------------------------------------------------------
# the boundary: model(batch)
# ----------------------------------------------------------------------------------------------
@torch.no_grad()
def generate(sd, param, batch, search='greedy', max_steps=40, cached=True, trace=None, taps=None,
             raw_trace=None):
    """CaptioningModel.forward -> forward_one -> infer (layers/decoder.py:838-877, 977-1011).

    batch: {'image': Tensor | list[Tensor], 'prefix'?: Long[1,P]} -> {'predictions','logprobs'}.
    raw_trace (list) receives the raw `decoding_step` output [rows, V] of every step; trace the
    search loop's view (greedy: after no-repeat / EOS forcing)."""
    feats = visual_features(sd, param, batch['image'])
    if taps is not None:
        taps['visual_features'] = feats
    B = feats.shape[0]
    if 'prefix' in batch:
        assert len(batch['prefix']) == 1 and B == 1, 'not supported'            # :985-989
        start = batch['prefix'].long()
    else:
        start = torch.full((B, 1), CLS, dtype=torch.long)
    beam = 1 if search == 'greedy' else 4
    if cached:
        dec = CachedDecoder(sd, feats, beam=beam, taps=taps)

        def step_fn(partial):
            return dec.feed(partial[:, dec.n_text:])
        reorder = dec.reorder
    else:
        def step_fn(partial):
            return as_shipped_step(sd, feats, partial)
        reorder = None

    def step(partial):
        z = step_fn(partial)
        if raw_trace is not None:
            raw_trace.append(z.clone())
        return z
    if search == 'greedy':
        pred, lp = greedy_search(start, step, max_steps=max_steps, trace=trace)
    elif search == 'beam':
        pred, lp = beam_search(start, step, reorder=reorder, max_steps=max_steps, trace=trace)
    else:
        raise ValueError(search)
    if 'prefix' in batch:
        pred = pred[:, start.shape[1]:]                                          # :1004-1006
    return {'predictions': pred, 'logprobs': lp}
