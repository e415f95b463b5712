"""The caption generator of the open-vocabulary head (SURVEY.md section 8 row f4): `CaptionTransformer`
(open_set/models/transformers/caption_tranformer.py:20-43: adapter, sinusoidal positions, 4 post-norm decoder blocks of
masked self-attention / cross-attention over the query embeddings / FFN, open_set/models/transformers/transformers.py
:58-134, :180-234, :252-267, and the 30 522-way generator), its training loss (`loss_caption_generation`,
open_set/models/mask2former_head.py:552-583) and the test-time beam search (open_set/utils/eval/inference.py:84-157).

The module carries the reference's state_dict keys (checkpoints load unchanged); its forward AND backward are the stage
kernels of the C-ABI library through the autograd nodes of train.py -- every linear layer a `cgg_gemm_f32` call (tcgen05
kind::tf32 in the tf32 training mode, fp32 FMA otherwise), the attention as the (image, head)-batched products with the
row-softmax kernels (`_AttentionViews`: 8 heads x 96, causal + key-padding masks as a bitmap), LayerNorm, broadcast adds.
The beam search (`beam_search_batch`) runs every image of a batch at once on the device: the network in fp32 FMA mode with
the self-attention keys / values of earlier tokens cached per beam, and the reference's candidate bookkeeping (top-k
over the flattened beams, finished list, max_idx) in the kernels of csrc/caption_kernels.cu, so that each image's token
sequences are the ones the reference's search produces for it alone."""
import math

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import lib as _lib
from .train import _K, _Linear, _LayerNorm, _AddRows, _AttentionViews, _p

BOS_TOKEN, EOS_TOKEN = 101, 102             # bert-base-uncased [CLS] / [SEP] (mask2former_head.py:30-31)


class _SelfAttn(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.qkv_layer = nn.Linear(dim, 3 * dim)
        self.out_layer = nn.Linear(dim, dim)


class _CrossAttn(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.to_qry, self.to_key, self.to_val, self.to_out = (nn.Linear(dim, dim) for _ in range(4))


class _FFN(nn.Module):
    """FeedForwardNetwork([in, ff, in], [ReLU, Identity], [drop, 0]): keys linears.{0,1}.0.*"""

    def __init__(self, dim, ff, drop):
        super().__init__()
        self.linears = nn.ModuleList([
            nn.Sequential(nn.Linear(dim, ff), nn.Dropout(drop) if drop > 0.0 else nn.Identity(), nn.ReLU()),
            nn.Sequential(nn.Linear(ff, dim), nn.Identity(), nn.Identity())])


class _Block(nn.Module):
    def __init__(self, dim, ff, heads, drop, pre_norm):
        super().__init__()
        self.mha_layer, self.crx_layer, self.ffn_layer = _SelfAttn(dim), _CrossAttn(dim), _FFN(dim, ff, drop)
        self.dropout_layer = nn.ModuleDict({k: nn.Dropout(drop) for k in ('mha', 'crx', 'ffn')})
        self.layer_normalz = nn.ModuleDict({
            k: nn.ModuleList([nn.LayerNorm(dim) if pre_norm else nn.Identity(),
                              nn.LayerNorm(dim) if not pre_norm else nn.Identity()]) for k in ('mha', 'crx', 'ffn')})


class _Decoder(nn.Module):
    def __init__(self, n, dim, ff, heads, drop, pre_norm):
        super().__init__()
        self.decoders = nn.ModuleList([_Block(dim, ff, heads, drop, pre_norm) for _ in range(n)])


class _Positions(nn.Module):
    """PositionalEncoding (transformers.py:9-25): sin on even, cos on odd channels of pos / 10000^((j - j%2)/dim)."""

    def __init__(self, seq_length, dim, drop):
        super().__init__()
        pos = np.arange(0, seq_length)[:, None]
        idx = np.fromfunction(lambda _, j: j - j % 2, shape=(1, dim))
        mask = np.fromfunction(lambda _, j: j % 2 == 0, shape=(1, dim))
        pnt = pos / (10000 ** (idx / dim))
        self.register_buffer('psne_layer', torch.tensor(np.sin(pnt) * mask + np.cos(pnt) * (1 - mask)).float())
        self.drop_layer = nn.Dropout(drop)


def _pack_bits(mask):
    """(B, Lq, Lk) bool (True = excluded) -> (B, Lq, ceil(Lk/32)) int32 words, bit i of word w = key 32 w + i."""
    B, Lq, Lk = mask.shape
    W = (Lk + 31) // 32
    m = torch.zeros((B, Lq, W * 32), dtype=torch.int64, device=mask.device)
    m[:, :, :Lk] = mask.long()
    words = (m.view(B, Lq, W, 32) << torch.arange(32, device=mask.device)).sum(-1)
    return (words & 0xffffffff).to(torch.int64).sub_((words >> 31 & 1) << 32).to(torch.int32).contiguous()


class CaptionTransformerB200(nn.Module):
    """Constructor arguments and state_dict keys of `CaptionTransformer` (caption_tranformer.py:20-36)."""

    def __init__(self, nb_layers, input_dim, hidden_dim, ff_dim, nb_heads, drop_val, pre_norm, seq_length, nb_tokens, **kw):
        super().__init__()
        assert hidden_dim % nb_heads == 0 and (hidden_dim // nb_heads) % 4 == 0
        self.nb_heads, self.hidden_dim, self.pre_norm = nb_heads, hidden_dim, pre_norm
        self.adapter = nn.Linear(input_dim, hidden_dim) if input_dim != hidden_dim else nn.Identity()
        self.position_encoder = _Positions(seq_length, hidden_dim, drop_val)
        self.transformer_decoder = _Decoder(nb_layers, hidden_dim, ff_dim, nb_heads, drop_val, pre_norm)
        self.generator = nn.Linear(hidden_dim, nb_tokens)
        self._kern = None            # (runtime owner, tf32 flag): set by the head

    # ---- plumbing
    def bind(self, head):
        self._head = [head]          # in a list: not a submodule

    def _k(self, device, exact):
        head = self._head[0]
        tf32 = (not exact) and head.train_precision == 'tf32' and torch.is_grad_enabled()
        return _K(head._runtime(device), tf32=tf32)

    def forward(self, tgt, memory, tgt_mask=None, memory_mask=None, tgt_key_padding_mask=None, memory_key_padding_mask=None,
                exact=False):
        """tgt (B, L, hidden) token embeddings, memory (B, Q, input_dim) query embeddings; tgt_key_padding_mask (B, L) bool
        (True = padding).  Returns (list of the nb_layers block outputs (B, L, hidden), logits of the last one (B, L, vocab))
        like caption_tranformer.py:38-43.  `exact`: fp32 FMA contractions whatever the training precision (beam search)."""
        if memory_mask is not None or memory_key_padding_mask is not None or tgt_mask is not None:
            raise _lib.CggError('only the causal tgt mask + tgt_key_padding_mask form the reference uses is built')
        if memory.shape[0] != tgt.shape[0]:
            raise _lib.CggError('memory has %d images, tgt %d' % (memory.shape[0], tgt.shape[0]))
        if not tgt.is_cuda:
            raise _lib.CggError('the caption transformer runs on CUDA only (no CPU fallback)')
        k = self._k(tgt.device, exact)
        B, L, C = tgt.shape
        Q = memory.shape[1]
        H, d = self.nb_heads, C // self.nb_heads
        scale = 1.0 / math.sqrt(d)
        active = lambda m: self.training and isinstance(m, nn.Dropout) and m.p > 0                         # noqa: E731
        drop = lambda x, m: m(x) if active(m) else x                                                       # noqa: E731
        lin = lambda x, m, res=None, relu=False: _Linear.apply(k, x, m.weight, m.bias, res, 1.0, relu)     # noqa: E731
        # residual + projection: fused into the GEMM epilogue unless a dropout sits between them (training with drop_val > 0)
        proj = lambda o, m, res, dl: (res + drop(lin(o, m), dl)) if active(dl) else lin(o, m, res=res)      # noqa: E731
        ln = lambda x, m: x if isinstance(m, nn.Identity) else _LayerNorm.apply(k, x, m.weight, m.bias, m.eps)   # noqa: E731
        mem = memory.float().contiguous().view(B * Q, -1)
        if not isinstance(self.adapter, nn.Identity):
            mem = lin(mem, self.adapter)
        x = _AddRows.apply(k, tgt.float().contiguous(), self.position_encoder.psne_layer[:L].contiguous(), B)
        x = drop(x, self.position_encoder.drop_layer).view(B * L, C)
        # causal mask (build_mask: key j > query i excluded) + key padding, as the attention kernels' bitmap
        causal = torch.ones((L, L), dtype=torch.bool, device=tgt.device).triu(1)[None].expand(B, L, L)
        if tgt_key_padding_mask is not None:
            causal = causal | tgt_key_padding_mask.bool()[:, None, :]
        self_bits = _pack_bits(causal)
        outs = []
        for blk in self.transformer_decoder.decoders:
            nz = blk.layer_normalz
            # masked self-attention (transformers.py:102-134): fused qkv, per head [q | k | v] of 3*d columns
            tmp = ln(x, nz['mha'][0])
            qkv = lin(tmp, blk.mha_layer.qkv_layer).view(B, L, H, 3, d)
            o = _AttentionViews.apply(k, qkv[:, :, :, 0], qkv[:, :, :, 1], qkv[:, :, :, 2], self_bits, None, scale)
            x = ln(proj(o.view(B * L, C), blk.mha_layer.out_layer, tmp, blk.dropout_layer['mha']), nz['mha'][1])
            # cross-attention over the (adapted) query embeddings (:58-100)
            tmp = ln(x, nz['crx'][0])
            ca = blk.crx_layer
            q4 = lin(tmp, ca.to_qry).view(B, L, H, d)
            k4 = lin(mem, ca.to_key).view(B, Q, H, d)
            v4 = lin(mem, ca.to_val).view(B, Q, H, d)
            o = _AttentionViews.apply(k, q4, k4, v4, None, None, scale)
            x = ln(proj(o.view(B * L, C), ca.to_out, tmp, blk.dropout_layer['crx']), nz['crx'][1])
            # FFN (:27-56; note the reference feeds `agg`, not the pre-normed tmp, :229)
            tmp = ln(x, nz['ffn'][0])
            f0, f1 = blk.ffn_layer.linears[0], blk.ffn_layer.linears[1]
            if self.training and isinstance(f0[1], nn.Dropout):
                h = F.relu(f0[1](lin(x, f0[0])))                       # Linear -> Dropout -> ReLU
            else:
                h = lin(x, f0[0], relu=True)
            x = ln(proj(h, f1[0], tmp, blk.dropout_layer['ffn']), nz['ffn'][1])
            outs.append(x.view(B, L, C))
        logits = lin(x, self.generator).view(B, L, -1)
        return outs, logits


def caption_generation_loss(head, cls_emb_preds, gt_caption_ids_list, gt_caption_embs_list, gt_caption_mask_list,
                            gt_caption_nouns_ids_list=None, loss_weight=2.0):
    """loss_caption_generation of one head call (mask2former_head.py:552-583): teacher-forced next-token cross entropy of
    the caption transformer over the query embeddings, ignore_index 0, mean over all B*(T-1) positions."""
    embs = torch.stack(list(gt_caption_embs_list), 0)
    masks = torch.stack(list(gt_caption_mask_list), 0).bool()
    logits = head.caption_generator(tgt=embs[:, :-1, :], memory=cls_emb_preds,
                                    tgt_key_padding_mask=torch.logical_not(masks[:, :-1]))[1].flatten(0, 1)
    ids_list = [t.clone() for t in gt_caption_ids_list]
    if head.gen_only_obj_nouns or head.gen_mask_obj_nouns or head.gen_replace_obj_nouns:      # :563-579, host-side like the reference
        for i, ids in enumerate(ids_list):
            nouns = gt_caption_nouns_ids_list[i].cpu().numpy().tolist()
            for j in range(len(ids)):
                if int(ids[j]) not in nouns:
                    if head.gen_only_obj_nouns:
                        ids[j] = 0
                else:
                    if head.gen_mask_obj_nouns:
                        ids[j] = 0
                        break
                    if head.gen_replace_obj_nouns:
                        ids[j] = 4874
    gt = torch.stack(ids_list, 0)[:, 1:].flatten(0, 1).long()
    from .matching import _WeightedCE
    cw = torch.ones((logits.shape[1],), dtype=torch.float32, device=logits.device)
    cw[0] = 0.0                                                       # ignore_index = 0: those rows contribute nothing
    row_loss, _ = _WeightedCE.apply(logits, gt, cw)
    return loss_weight * row_loss.sum() / gt.numel()


def _pow32(x, alpha):
    """x ** alpha as the reference applies it to an fp32 tensor: the power in double, rounded to fp32."""
    return float(np.float32(x ** alpha))


@torch.no_grad()
def _search_device(head, memory, BOS, EOS, max_len, beam_width, alpha):
    """Issues the batched search on the current stream without waiting for the device.  Every step runs all B * W rows:
    the new token's embedding, the decoder blocks with the self-attention keys / values of earlier positions cached per
    beam, the generator on every block's output, the beam scores and the selection.  The host reads the done-image count
    back asynchronously and stops issuing steps once it sees every image done.  Returns (state tensors, steps issued)."""
    gen = head.caption_generator
    psne = gen.position_encoder.psne_layer
    npos = psne.shape[0]
    if memory.dim() != 3 or memory.shape[0] < 1:
        raise _lib.CggError('memory must be (B, Q, dim) with B >= 1')
    if not 1 <= beam_width <= 32:
        raise _lib.CggError('beam_width must be in 1..32')
    if not 1 <= max_len <= npos:
        raise _lib.CggError('max_len must be in 1..%d (the position table)' % npos)
    if not memory.is_cuda:
        raise _lib.CggError('the caption beam search runs on CUDA only (no CPU fallback)')
    dev = memory.device
    k = gen._k(dev, True)
    blocks = gen.transformer_decoder.decoders
    B, Q, W = memory.shape[0], memory.shape[1], beam_width
    nb, D, H = len(blocks), gen.hidden_dim, gen.nb_heads
    d, n = D // H, B * W
    scale = 1.0 / math.sqrt(d)
    # the BOS step, then passes while a beam may continue (length + 1 < max_len - 1): pass s sees sequences of length s + 1
    steps = max(2, max_len - 2)
    T = steps + 1                                                   # the longest sequence, EOS included
    lin = lambda x, m, res=None, relu=False: _Linear.apply(k, x, m.weight, m.bias, res, 1.0, relu)     # noqa: E731
    ln = lambda x, m: x if isinstance(m, nn.Identity) else _LayerNorm.apply(k, x, m.weight, m.bias, m.eps)   # noqa: E731
    mem = memory.float().contiguous().view(B * Q, -1)
    if not isinstance(gen.adapter, nn.Identity):
        mem = lin(mem, gen.adapter)
    # cross-attention keys / values: once per image and block, shared by the image's beams
    kv_mem = [(lin(mem, b.crx_layer.to_key).view(B, Q, H, d), lin(mem, b.crx_layer.to_val).view(B, Q, H, d)) for b in blocks]
    cache = [k.new(nb, 2, n, steps, D) for _ in range(2)]          # double-buffered (block, k / v, row, position, D)
    i32 = dict(dtype=torch.int32, device=dev)
    st = dict(tokens=torch.full((B, W, T), BOS, **i32), weights=k.new(B, W).zero_(), n_active=torch.zeros(B, **i32),
              parent=torch.zeros((B, W), **i32), next_ids=torch.full((B, W), BOS, dtype=torch.int64, device=dev),
              fin_tokens=torch.zeros((B, W, T), **i32), fin_len=torch.zeros((B, W), **i32), fin_score=k.new(B, W).zero_(),
              n_fin=torch.zeros(B, **i32), max_idx=torch.zeros(B, **i32), done=torch.zeros(B, **i32),
              n_done=torch.zeros(1, **i32))
    state = _lib.BeamState(token_cap=T, **{name: t.data_ptr() for name, t in st.items()})
    cand_val, cand_col = k.new(n, W), torch.empty((n, W), **i32)
    n_done = torch.zeros(steps, dtype=torch.int32, pin_memory=True)
    events, checked = [], 0
    be = head.bert_embeddings
    for s in range(steps):
        x = head.extract_word_embeddings(be.word_embeddings.weight, be.LayerNorm.weight, be.LayerNorm.bias,
                                         st['next_ids'].view(n), eps=be.LayerNorm.eps)
        x = _AddRows.apply(k, x.view(n, 1, D), psne[s:s + 1], n).view(n, D)
        kc = cache[s % 2]
        outs = []
        for i, blk in enumerate(blocks):
            nz, ca = blk.layer_normalz, blk.crx_layer
            tmp = ln(x, nz['mha'][0])
            qkv = lin(tmp, blk.mha_layer.qkv_layer)
            o = k.new(n, D)
            k.chk(k.lib.cgg_caption_self_attn_step(k.h, _p(qkv), _p(kc[i, 0]), _p(kc[i, 1]), _p(o), n, H, d, s, steps, scale,
                                                   k.s()), 'cgg_caption_self_attn_step')
            x = ln(lin(o, blk.mha_layer.out_layer, res=tmp), nz['mha'][1])
            tmp = ln(x, nz['crx'][0])
            o = _AttentionViews.apply(k, lin(tmp, ca.to_qry).view(B, W, H, d), kv_mem[i][0], kv_mem[i][1], None, None, scale)
            x = ln(lin(o.view(n, D), ca.to_out, res=tmp), nz['crx'][1])
            tmp = ln(x, nz['ffn'][0])
            f0, f1 = blk.ffn_layer.linears[0], blk.ffn_layer.linears[1]
            x = ln(lin(lin(x, f0[0], relu=True), f1[0], res=tmp), nz['ffn'][1])
            outs.append(x)
        logits = lin(torch.stack(outs, 0).view(nb * n, D), gen.generator)        # the generator on every block's rows
        first, length = int(s == 0), s + 1
        pw, pw1 = _pow32(length, alpha), _pow32(length + 1, alpha)
        k.chk(k.lib.cgg_caption_beam_scores(k.h, _p(logits), nb, B, W, logits.shape[1], first, state, pw,
                                            _p(cand_val), _p(cand_col), k.s()), 'cgg_caption_beam_scores')
        k.chk(k.lib.cgg_caption_beam_select(k.h, _p(cand_val), _p(cand_col), B, W, first, length, max_len, npos, pw, pw1,
                                            EOS, state, k.s()), 'cgg_caption_beam_select')
        if s + 1 < steps:
            k.chk(k.lib.cgg_caption_cache_reorder(k.h, _p(kc), _p(cache[(s + 1) % 2]), _p(st['parent']), nb, B, W, steps,
                                                  s + 1, D, k.s()), 'cgg_caption_cache_reorder')
        n_done[s].copy_(st['n_done'][0], non_blocking=True)
        events.append(torch.cuda.Event())
        events[-1].record(torch.cuda.current_stream(dev))
        while checked <= s and events[checked].query():
            if int(n_done[checked]) == B:
                return st, s + 1
            checked += 1
    return st, steps


def _search_results(st, tokenizer=None):
    """The one synchronisation of a search: its state as one dict per image (the shape `beam_search` returns)."""
    torch.cuda.current_stream(st['n_fin'].device).synchronize()
    n_fin, max_idx = st['n_fin'].tolist(), st['max_idx'].tolist()
    fin_len, fin_tokens, fin_score = st['fin_len'].tolist(), st['fin_tokens'].cpu(), st['fin_score'].tolist()
    results = []
    for b in range(len(n_fin)):
        finished = [(fin_tokens[b, j, :fin_len[b][j]].tolist(), fin_score[b][j]) for j in range(n_fin[b])]
        best = finished[max_idx[b]] if finished else (None, None)
        text = None
        if tokenizer is not None and finished:
            text = tokenizer.decode(best[0])[1:-1]                                           # inference.py:149-154
        results.append(dict(ids=best[0], score=best[1], finished=finished, text=text))
    return results


def beam_search_batch(head, memory, BOS=BOS_TOKEN, EOS=EOS_TOKEN, max_len=35, beam_width=7, alpha=0.7, tokenizer=None):
    """inference.py:84-157 for every image of memory (B, Q, dim) at once, on the device: one dict per image with the best
    sentence's token ids, its score, all finished (ids, score) pairs in the reference's order and, with a `tokenizer`
    (bert-base-uncased), the decoded sentence -- for each image what the reference's beam search returns for it alone."""
    st, _ = _search_device(head, memory, BOS, EOS, max_len, beam_width, alpha)
    return _search_results(st, tokenizer)


def beam_search(head, memory, BOS=BOS_TOKEN, EOS=EOS_TOKEN, max_len=35, beam_width=7, alpha=0.7, tokenizer=None):
    """The beam search of one image (memory (1, Q, dim)): `beam_search_batch(...)[0]`."""
    if memory.dim() != 3 or memory.shape[0] != 1:
        raise _lib.CggError('beam_search takes one image (memory (1, Q, dim)); use beam_search_batch for a batch')
    return beam_search_batch(head, memory, BOS, EOS, max_len, beam_width, alpha, tokenizer)[0]
