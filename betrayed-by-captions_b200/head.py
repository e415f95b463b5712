"""Host-side mirror of the reference's open-vocabulary Mask2Former head for the decoder hot path.

``Mask2FormerHeadOpenB200`` keeps the forward contract of ``Mask2FormerHeadOpen``
(open_set/models/mask2former_head.py:763-849): ``forward(feats, img_metas) ->
(cls_pred_list, cls_emb_pred_list, mask_pred_list)``, each of length num_layers+1, and accepts
the reference's state_dict keys unchanged (SURVEY.md section 8b), so a trained CGG checkpoint
loads into it with ``load_state_dict``.  Everything after ``self.pixel_decoder(feats)``
(head.py:787) runs in the CUDA library behind include/cgg_b200.h; PyTorch only owns memory
and the stream.  There is no torch/CPU fallback: without the built library or without a CUDA
device the forward raises.
"""
import ctypes as C
import math

import torch
import torch.nn as nn

from . import lib as _lib


class _Attn(nn.Module):
    """Parameter container with mmcv's key layout: attentions.<i>.attn.{in_proj_*,out_proj.*}."""

    def __init__(self, embed, heads):
        super().__init__()
        self.attn = nn.MultiheadAttention(embed, heads, 0.0)


class _FFN(nn.Module):
    """mmcv FFN key layout: ffns.0.layers.0.0.* and ffns.0.layers.1.*"""

    def __init__(self, embed, ffn):
        super().__init__()
        self.layers = nn.Sequential(nn.Sequential(nn.Linear(embed, ffn), nn.ReLU(inplace=True), nn.Dropout(0.0)),
                                    nn.Linear(ffn, embed), nn.Dropout(0.0))


class _Layer(nn.Module):
    def __init__(self, embed, heads, ffn):
        super().__init__()
        self.attentions = nn.ModuleList([_Attn(embed, heads), _Attn(embed, heads)])  # 0 = cross, 1 = self
        self.ffns = nn.ModuleList([_FFN(embed, ffn)])
        self.norms = nn.ModuleList([nn.LayerNorm(embed) for _ in range(3)])


class _Decoder(nn.Module):
    def __init__(self, num_layers, embed, heads, ffn):
        super().__init__()
        self.layers = nn.ModuleList([_Layer(embed, heads, ffn) for _ in range(num_layers)])
        self.post_norm = nn.LayerNorm(embed)
        self.embed_dims = embed


def _get(cfg, *path, default=None):
    for p in path:
        if cfg is None:
            return default
        cfg = cfg.get(p) if isinstance(cfg, dict) else getattr(cfg, p, None)
    return default if cfg is None else cfg


class _BertEmbeddings(nn.Module):
    """open_set/models/utils/bert_embeddings.py:4-13: only the word-embedding table and the embedding LayerNorm of
    bert-base-uncased (state_dict keys bert_embeddings.word_embeddings.weight, bert_embeddings.LayerNorm.*); frozen."""

    def __init__(self, vocab=30522, d=768, eps=1e-12):
        super().__init__()
        self.word_embeddings = nn.Embedding(vocab, d, padding_idx=0)
        self.LayerNorm = nn.LayerNorm(d, eps=eps)
        for p_ in self.parameters():
            p_.requires_grad = False


class Mask2FormerHeadOpenB200(nn.Module):
    """Drop-in for ``Mask2FormerHeadOpen`` on the decoder hot path.

    Constructor kwargs follow the reference (head.py:76-100 and init_kwargs :175-195); the ones
    that only matter to losses / caption generation are accepted and ignored.  New kwargs:
    ``precision`` ('fp32' parity mode | 'bf16' throughput mode), ``train_precision`` ('fp32' | 'tf32', the arithmetic
    of the training step's contractions; default follows ``precision``), ``cuda_graph`` (replay the whole path
    as one CUDA graph per set of input buffers) and ``pixel_decoder`` may be an
    ``nn.Module`` instance (mmdet builds it from the config dict in the real stack, see
    INTEGRATION.md)."""

    def __init__(self, in_channels=None, feat_channels=256, out_channels=256, num_things_classes=80,
                 num_stuff_classes=53, num_queries=100, num_transformer_feat_level=3, pixel_decoder=None,
                 enforce_decoder_input_project=False, transformer_decoder=None, positional_encoding=None,
                 precision='fp32', d_lang=768, cuda_graph=False, final_mask_only=False, **kwargs):
        super().__init__()
        self.cuda_graph = bool(cuda_graph)
        # inference shortcut (opt-in, bf16 mode): only the last head call's mask logits are produced; the mask list
        # then holds None for the intermediate head calls (only [-1] is consumed at test time, head.py:943-945)
        self.final_mask_only = bool(final_mask_only)
        if num_transformer_feat_level != 3:
            raise ValueError('the B200 path is built for 3 feature levels (1/32, 1/16, 1/8)')
        if enforce_decoder_input_project or feat_channels != out_channels:
            raise ValueError('decoder_input_projs must be Identity (feat_channels == embed dims, head.py:125-131)')
        self.num_things_classes, self.num_stuff_classes = num_things_classes, num_stuff_classes
        self.num_classes = num_things_classes + num_stuff_classes
        self.num_queries = num_queries
        self.num_transformer_feat_level = 3
        self.num_heads = _get(transformer_decoder, 'transformerlayers', 'attn_cfgs', 'num_heads', default=8)
        self.num_transformer_decoder_layers = _get(transformer_decoder, 'num_layers', default=9)
        ffn = _get(transformer_decoder, 'transformerlayers', 'feedforward_channels', default=2048)
        self.feat_channels = feat_channels
        self.ffn_channels = ffn
        self.d_lang = d_lang
        self.precision = precision
        self.softmax_temperature = kwargs.get('softmax_temperature', 10.0)
        # head.py:178,739-744: without class embeddings there is no v2l_transform / class_embs, the embedding
        # prediction IS the class prediction and pred_emb_norm is never applied (the class-agnostic pre-training
        # configs coco_ag_pretrain_3x.py / p20_ag_pretrain.py run this way)
        self.use_class_emb = bool(kwargs.get('use_class_emb', False))
        self.pred_emb_norm = kwargs.get('pred_emb_norm', False)
        # training-step arithmetic: 'fp32' (FMA, the parity mode with gradients) or 'tf32' (every contraction on tcgen05
        # kind::tf32 MMAs straight from the fp32 tensors; softmax, LayerNorm and all accumulation stay fp32)
        self.train_precision = kwargs.get('train_precision', 'tf32' if precision == 'bf16' else 'fp32')
        if self.train_precision not in ('fp32', 'tf32'):
            raise ValueError("train_precision must be 'fp32' or 'tf32'")
        # weight / bias gradients of the linear layers accumulated straight into the .grad tensors on a side stream
        # (train._WgradSide): True = for parameters managed by a train.GradReducer, 'always' = whenever .grad exists at
        # forward time, False = never (everything through autograd)
        self.fused_wgrad = kwargs.get('fused_wgrad', True)
        self.text_emb_norm = kwargs.get('text_emb_norm', True)
        self.pixel_decoder = pixel_decoder if isinstance(pixel_decoder, nn.Module) else None
        # ---- parameters under the reference's names
        self.transformer_decoder = _Decoder(self.num_transformer_decoder_layers, feat_channels, self.num_heads, ffn)
        self.query_embed = nn.Embedding(num_queries, feat_channels)
        self.query_feat = nn.Embedding(num_queries, feat_channels)
        self.level_embed = nn.Embedding(3, feat_channels)
        self.cls_embed = nn.Linear(feat_channels, self.num_classes + 1)
        self.mask_embed = nn.Sequential(nn.Linear(feat_channels, feat_channels), nn.ReLU(inplace=True),
                                        nn.Linear(feat_channels, feat_channels), nn.ReLU(inplace=True),
                                        nn.Linear(feat_channels, out_channels))
        if self.use_class_emb:
            self.v2l_transform = nn.Linear(feat_channels, d_lang)
            self.register_buffer('class_embs', torch.zeros(self.num_classes + 1, d_lang))
        # caption side (head.py:249-254, :171): frozen BERT word embeddings for the noun tokens, grounding-loss weight
        self.use_caption = bool(kwargs.get('use_caption', False))
        self.caption_emb_type = kwargs.get('caption_emb_type', 'bert')
        self.loss_only_last = bool(kwargs.get('loss_only_last', False))
        self.loss_aux_weight = float(kwargs.get('loss_aux_weight', 1.0))
        self.loss_grounding_weight = float(_get(kwargs.get('loss_grounding'), 'loss_weight', default=1.0))
        self.test_cfg = kwargs.get('test_cfg') or {}
        self.bert_embeddings = None
        if self.use_caption:
            if self.caption_emb_type != 'bert':
                raise ValueError('only caption_emb_type="bert" is built (the shipped configs use it)')
            self.bert_embeddings = _BertEmbeddings(kwargs.get('bert_vocab_size', 30522), d_lang)
        # caption generator (head.py:246-248, configs .../coco_panoptic_p20.py:100-110): CaptionTransformer over the query
        # embeddings, its loss and the test-time beam search (row f4, cgg_b200/caption.py)
        self.use_caption_generation = bool(kwargs.get('use_caption_generation', False))
        self.gen_only_obj_nouns = bool(kwargs.get('gen_only_obj_nouns', False))
        self.gen_mask_obj_nouns = bool(kwargs.get('gen_mask_obj_nouns', False))
        self.gen_replace_obj_nouns = bool(kwargs.get('gen_replace_obj_nouns', False))
        self.loss_caption_generation_weight = float(_get(kwargs.get('loss_caption_generation'), 'loss_weight', default=1.0))
        self.caption_generator = None
        self.tokenizer = None          # optional bert-base-uncased tokenizer: simple_test(with_caption) then returns text
        cg = kwargs.get('caption_generator')
        if cg:
            from .caption import CaptionTransformerB200
            cg = {k_: v for k_, v in dict(cg).items() if k_ != 'type'}
            self.caption_generator = CaptionTransformerB200(**cg)
            self.caption_generator.bind(self)
            if self.bert_embeddings is None:        # the generator reads token embeddings (caption_gen_emb_type 'bert')
                self.bert_embeddings = _BertEmbeddings(kwargs.get('bert_vocab_size', 30522), d_lang)
        # head.py:151-158: with a train_cfg the reference builds its assigner / sampler / point-sampling parameters; here
        # that is the MatchingLosses object behind `loss()` (row f2: Hungarian targets, class and point-sampled mask losses)
        self.train_cfg = kwargs.get('train_cfg') or None
        if self.train_cfg:
            from .matching import MatchingLosses
            self.matching_losses = MatchingLosses(self, train_cfg=self.train_cfg, loss_cls=kwargs.get('loss_cls'),
                                                  loss_cls_emb=kwargs.get('loss_cls_emb'), loss_mask=kwargs.get('loss_mask'),
                                                  loss_dice=kwargs.get('loss_dice'))
        self._rt = None
        self.init_weights()

    def init_weights(self):
        """head.py:231-240: xavier_normal_ on every >=2-D transformer-decoder parameter."""
        for p in self.transformer_decoder.parameters():
            if p.dim() > 1:
                nn.init.xavier_normal_(p)

    # ------------------------------------------------------------------ runtime plumbing
    def _runtime(self, device):
        if self._rt is None or self._rt.device != device:
            self._rt = _Runtime(self, device)
        return self._rt

    def decoder_forward(self, mask_features, multi_scale_memorys, return_debug=False):
        """The seam that is replaced: head.py:787 (exclusive) .. :849.  Returns the three lists
        (and, with return_debug, the decoder states / attention-mask bitmaps / fallback flags)."""
        if not mask_features.is_cuda:
            raise _lib.CggError('Mask2FormerHeadOpenB200 runs on CUDA only (no CPU fallback)')
        rt = self._runtime(mask_features.device)
        return rt.forward(mask_features, list(multi_scale_memorys), return_debug)

    def forward(self, feats, img_metas):
        batch_size = len(img_metas)
        if self.pixel_decoder is None:
            raise _lib.CggError('no pixel_decoder module attached (it is the step before the path and stays '
                                'mmdet\'s MSDeformAttnPixelDecoder)')
        mask_features, multi_scale_memorys = self.pixel_decoder(feats)       # head.py:787
        assert mask_features.shape[0] == batch_size
        return self.decoder_forward_auto(mask_features, multi_scale_memorys)

    def decoder_forward_auto(self, mask_features, multi_scale_memorys):
        """Inference kernels under no_grad, the autograd-connected training path (train.py) when gradients are
        being recorded -- the reference's forward is one function for both (head.py:763-849)."""
        if torch.is_grad_enabled() and (mask_features.requires_grad or any(p.requires_grad for p in self.parameters())):
            from .train import decoder_forward_train
            return decoder_forward_train(self, mask_features, multi_scale_memorys)
        with torch.no_grad():
            return self.decoder_forward(mask_features, multi_scale_memorys)

    # -------------------------------------------------------------- grounding-side helpers
    def _get_cls_emb_logits(self, cls_emb_preds):
        """head.py:631-648."""
        from .grounding import similarity
        B, Q, D = cls_emb_preds.shape
        return similarity(cls_emb_preds.reshape(B * Q, D), self.class_embs,
                          1.0 / float(self.softmax_temperature)).view(B, Q, -1)

    def test_time_att(self, mask_cls_emb_results, nouns_embs):
        """simple_test `att`, head.py:973-978."""
        rt = self._runtime(mask_cls_emb_results.device)
        return rt.similarity(mask_cls_emb_results[0], nouns_embs, 1.0)

    def extract_word_embeddings(self, table, ln_weight, ln_bias, ids, eps=1e-12):
        """head.py:686-698 (bert branch) for a stacked (B, max_tokens) id tensor."""
        rt = self._runtime(ids.device)
        return rt.noun_embeddings(table, ln_weight, ln_bias, ids, eps, self.text_emb_norm)

    def extract_caption_embeddings(self, ids_list, mask_list):
        """The reference's `extract_word_embeddings(ids_list, mask_list, 'bert')` (head.py:686-709): per image, the BERT
        word-embedding rows of the caption's noun ids, LayerNorm'ed when text_emb_norm.  Returns (embs_list, mask_list)."""
        if self.bert_embeddings is None:
            raise _lib.CggError('the head was built without use_caption=True: no BERT embedding table')
        be = self.bert_embeddings
        ids = torch.stack(list(ids_list), 0)
        embs = self.extract_word_embeddings(be.word_embeddings.weight, be.LayerNorm.weight, be.LayerNorm.bias, ids,
                                            eps=be.LayerNorm.eps)
        return list(embs.unbind(0)), list(mask_list)

    # ------------------------------------------------------------------- the reference's callers
    def loss(self, all_cls_scores, all_cls_emb_preds, all_mask_preds, gt_labels_list, gt_masks_list, gt_caption_ids_list,
             gt_caption_embs_list, gt_caption_mask_list, gt_caption_nouns_ids_list, gt_caption_nouns_embs_list,
             gt_caption_nouns_mask_list, img_metas):
        """head.py:393-462 for the term that is on the path: the caption-grounding loss of every head call
        (loss_single :540-548), computed on the CUDA kernels with the batched cross-rank gather, merged with the
        matching-based terms (loss_cls / loss_cls_emb / loss_mask / loss_dice: Hungarian assignment on point-sampled masks,
        :320-390, :591-627 -- the step AFTER the path, SURVEY.md 8f rank 2) from `self.matching_losses`
        (cgg_b200/matching.py `MatchingLosses`, built by the constructor when a train_cfg is given; any callable
        `(all_cls_scores, all_cls_emb_preds, all_mask_preds, gt_labels_list, gt_masks_list, img_metas) -> dict` works)."""
        from .grounding import gather_captions_and_preds, grounding_loss
        losses = {}
        if self.use_caption:
            preds = torch.stack(list(all_cls_emb_preds), 0)                       # (L+1, B, Q, d_l)
            embs, mask, preds_all = gather_captions_and_preds(gt_caption_nouns_embs_list, gt_caption_nouns_mask_list, preds)
            n = preds_all.shape[0]
            for j in range(n):
                if self.loss_only_last and j != n - 1:
                    continue
                lg = grounding_loss(preds_all[j], embs, mask, float(self.softmax_temperature), self.loss_grounding_weight)
                if j == n - 1:
                    losses['loss_grounding'] = lg
                else:
                    losses['d%d.loss_grounding' % j] = lg * self.loss_aux_weight
        if self.use_caption_generation:                                           # loss_single :550-583
            from .caption import caption_generation_loss
            n = len(all_cls_emb_preds)
            for j in range(n):
                if self.loss_only_last and j != n - 1:
                    continue
                lc = caption_generation_loss(self, all_cls_emb_preds[j], gt_caption_ids_list, gt_caption_embs_list,
                                             gt_caption_mask_list, gt_caption_nouns_ids_list,
                                             self.loss_caption_generation_weight)
                if j == n - 1:
                    losses['loss_caption_generation'] = lc
                else:
                    losses['d%d.loss_caption_generation' % j] = lc * self.loss_aux_weight
        hook = getattr(self, 'matching_losses', None)
        if hook is not None:
            losses.update(hook(all_cls_scores, all_cls_emb_preds, all_mask_preds, gt_labels_list, gt_masks_list, img_metas))
        return losses

    def forward_train(self, feats, img_metas, gt_bboxes, gt_labels, gt_masks, gt_semantic_seg, gt_caption_ids,
                      gt_caption_mask, gt_caption_nouns_ids, gt_caption_nouns_mask, gt_bboxes_ignore=None, **kwargs):
        """head.py:851-921 (same signature): forward on the autograd-connected path, noun embeddings, losses.
        mmdet's inputs (BitmapMasks, a gt_semantic_seg batch) go through `preprocess_gt` (:903) into compact targets; a
        list of dense mask tensors without a semantic map is passed to the losses as it is."""
        assert gt_bboxes_ignore is None
        if gt_masks is not None and (gt_semantic_seg is not None or not all(torch.is_tensor(m) for m in gt_masks)):
            gt_labels, gt_masks = self.preprocess_gt(gt_labels, gt_masks, gt_semantic_seg, img_metas)
        all_cls_scores, all_cls_emb_preds, all_mask_preds = self(feats, img_metas)
        nouns_embs = nouns_mask = cap_embs = None
        if self.use_caption_generation:                                                                 # :905-908
            cap_embs, gt_caption_mask = self.extract_caption_embeddings(gt_caption_ids, gt_caption_mask)
        if self.use_caption:
            nouns_embs, nouns_mask = self.extract_caption_embeddings(gt_caption_nouns_ids, gt_caption_nouns_mask)
        return self.loss(all_cls_scores, all_cls_emb_preds, all_mask_preds, gt_labels, gt_masks, gt_caption_ids, cap_embs,
                         gt_caption_mask, gt_caption_nouns_ids, nouns_embs, nouns_mask, img_metas)

    def preprocess_gt(self, gt_labels_list, gt_masks_list, gt_semantic_segs, img_metas):
        """mmdet 2.28.2 MaskFormerHead.preprocess_gt (head.py:903): per image, things labels then the stuff labels present
        in the semantic map (ascending) -> (labels_list, cgg_b200.matching.PanopticTargets).  The targets stay compact
        (unpadded things masks, the semantic map and its stuff labels on the device); the matching losses point-sample
        them as mmdet's dense padded int64 masks would be sampled."""
        from .matching import preprocess_gt
        return preprocess_gt(gt_labels_list, gt_masks_list, gt_semantic_segs, img_metas, self.num_things_classes,
                             self.num_stuff_classes, self.query_feat.weight.device)

    def simple_test(self, feats, img_metas, **kwargs):
        """head.py:923-980 (same signature and return tuple): last head call's outputs, masks upsampled to the padded
        input size, optional query x noun attention `att`, optional test-time label assignment (`gt_labels` / `gt_masks`:
        the Hungarian assignment of `_get_target_single`, cgg_b200/matching.py) and caption generation (`with_caption` /
        'cap_results': the beam search of cgg_b200/caption.py; the sentence text when `self.tokenizer` is set -- the
        reference downloads bert-base-uncased's tokenizer for that -- otherwise its token ids; for a batch of B > 1
        images, a list of B such results)."""
        from .postprocess import upsample_masks
        all_cls_scores, all_cls_emb_preds, all_mask_preds = self(feats, img_metas)
        mask_cls_results, mask_cls_emb_results, mask_pred_results = all_cls_scores[-1], all_cls_emb_preds[-1], all_mask_preds[-1]
        assigned_labels = mask_cls_results
        if kwargs.get('gt_labels', None) is not None:                                                  # :947-953
            from .grounding import similarity
            from .matching import MatchingLosses
            ml = getattr(self, 'matching_losses', None)
            if not isinstance(ml, MatchingLosses):
                ml = MatchingLosses(self, train_cfg=self.train_cfg)
            gl, gm = kwargs['gt_labels'][0][0], kwargs['gt_masks'][0][0]
            if torch.is_tensor(gm):
                gm = gm.to(mask_cls_results.device)
            else:                                    # mmdet BitmapMasks: compact things targets
                gl, gm = self.preprocess_gt([gl], [gm], None, img_metas[:1])
                gl = gl[0]
            logits = None
            if self.use_class_emb:
                logits = similarity(mask_cls_emb_results[0].float(), self.class_embs, 1.0 / float(self.softmax_temperature))
            assigned_labels = ml.get_target_single(mask_cls_results[0].float(), logits, mask_pred_results[0],
                                                   gl.to(mask_cls_results.device), gm)[0]
        img_shape = kwargs.get('img_shape') or img_metas[0]['batch_input_shape']
        mask_pred_results = upsample_masks(self, mask_pred_results, (img_shape[0], img_shape[1]))      # :957-964
        caption_generation_results = None
        if kwargs.get('with_caption', False) or 'cap_results' in self.test_cfg.get('eval_types', []):     # :966-970
            if self.caption_generator is None:
                raise _lib.CggError('with_caption needs a head built with caption_generator=dict(...)')
            from .caption import beam_search_batch
            res = beam_search_batch(self, mask_cls_emb_results.float(), max_len=35, beam_width=7, tokenizer=self.tokenizer)
            caption_generation_results = [r['text'] if self.tokenizer is not None else r['ids'] for r in res]
            if len(res) == 1:                          # one image: the reference's return value
                caption_generation_results = caption_generation_results[0]
        att = None
        if kwargs.get('with_att', False):                                                               # :973-978
            ids = kwargs['nouns_ids']
            be = self.bert_embeddings
            if be is None:
                raise _lib.CggError('with_att needs use_caption=True (BERT embedding table)')
            nouns_embs = self.extract_word_embeddings(be.word_embeddings.weight, be.LayerNorm.weight, be.LayerNorm.bias,
                                                      ids.reshape(-1), eps=be.LayerNorm.eps)
            att = self.test_time_att(mask_cls_emb_results, nouns_embs)
        return assigned_labels, mask_cls_emb_results, mask_pred_results, caption_generation_results, att

    def grounding_loss(self, cls_emb_pred, gt_caption_embs, gt_caption_mask, loss_weight=1.0):
        """losses/grounding_loss.py:9-77; differentiable w.r.t. cls_emb_pred (grounding.py)."""
        from .grounding import grounding_loss
        return grounding_loss(cls_emb_pred, gt_caption_embs, gt_caption_mask, float(self.softmax_temperature),
                              loss_weight)


def _ptr(t):
    return C.c_void_p(t.data_ptr())


class _Runtime:
    """One C-ABI handle + packed weight pointers + workspace for a head on one device."""

    def __init__(self, head, device):
        self.lib = _lib.load()
        self.head = head
        self.device = device
        self.handle = C.c_void_p()
        prec = {'fp32': _lib.FP32, 'bf16': _lib.BF16}[head.precision]
        self.d_lang = head.d_lang if head.use_class_emb else 0      # 0: no v2l_transform in the library either
        self.cfg = _lib.Config(head.num_queries, head.feat_channels, head.num_heads, head.ffn_channels,
                               head.num_transformer_decoder_layers, head.num_classes + 1, self.d_lang, prec,
                               int(bool(head.pred_emb_norm) and head.use_class_emb))
        with torch.cuda.device(device):
            _lib.check(self.lib.cgg_create(C.byref(self.handle), C.byref(self.cfg)), None, 'cgg_create')
        self.weights = None
        self.weights_key = None
        self.sizes = None
        self.workspace = None
        self.batch = None
        self._keep = []
        self._graphs = {}
        self._pos = {}

    def __del__(self):
        try:
            if self.handle:
                self.lib.cgg_destroy(self.handle)
        except Exception:
            pass

    # ---- weights
    def _pack_weights(self):
        h = self.head
        keep = []

        def f(t):
            t = t.detach()
            if t.dtype != torch.float32 or not t.is_contiguous() or t.device != self.device:
                t = t.to(device=self.device, dtype=torch.float32).contiguous()
            keep.append(t)
            return t.data_ptr()

        w = _lib.Weights()
        w.query_embed, w.query_feat, w.level_embed = f(h.query_embed.weight), f(h.query_feat.weight), f(h.level_embed.weight)
        w.cls_w, w.cls_b = f(h.cls_embed.weight), f(h.cls_embed.bias)
        for n, i in enumerate((0, 2, 4)):
            w.me_w[n], w.me_b[n] = f(h.mask_embed[i].weight), f(h.mask_embed[i].bias)
        if h.use_class_emb:
            w.v2l_w, w.v2l_b = f(h.v2l_transform.weight), f(h.v2l_transform.bias)
        w.post_norm_w, w.post_norm_b = f(h.transformer_decoder.post_norm.weight), f(h.transformer_decoder.post_norm.bias)
        for i, layer in enumerate(h.transformer_decoder.layers):
            lw = w.layers[i]
            ca, sa = layer.attentions[0].attn, layer.attentions[1].attn
            lw.cross_in_w, lw.cross_in_b = f(ca.in_proj_weight), f(ca.in_proj_bias)
            lw.cross_out_w, lw.cross_out_b = f(ca.out_proj.weight), f(ca.out_proj.bias)
            lw.self_in_w, lw.self_in_b = f(sa.in_proj_weight), f(sa.in_proj_bias)
            lw.self_out_w, lw.self_out_b = f(sa.out_proj.weight), f(sa.out_proj.bias)
            lw.ffn_w1, lw.ffn_b1 = f(layer.ffns[0].layers[0][0].weight), f(layer.ffns[0].layers[0][0].bias)
            lw.ffn_w2, lw.ffn_b2 = f(layer.ffns[0].layers[1].weight), f(layer.ffns[0].layers[1].bias)
            for n in range(3):
                lw.norm_w[n], lw.norm_b[n] = f(layer.norms[n].weight), f(layer.norms[n].bias)
        self.weights, self._keep = w, keep

    def _weights_key(self):
        return tuple((p.data_ptr(), p._version) for p in self.head.parameters())

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def prepare(self, H4, W4, level_sizes, batch):
        key = self._weights_key()
        sizes = (H4, W4, tuple(level_sizes))
        if self.weights is None or key != self.weights_key or sizes != self.sizes:
            self._pack_weights()
            lh = (C.c_int * 3)(*[s[0] for s in level_sizes])
            lw = (C.c_int * 3)(*[s[1] for s in level_sizes])
            _lib.check(self.lib.cgg_prepare(self.handle, C.byref(self.weights), H4, W4, lh, lw, self._stream()),
                       self.handle, 'cgg_prepare')
            self.weights_key, self.sizes = key, sizes
            self.batch = None
            self._graphs.clear()      # captured graphs bake in the handle's tables: stale after a re-prepare
        if self.batch != batch:
            self._graphs.clear()      # ... and the workspace pointer
            nbytes = self.lib.cgg_workspace_bytes(self.handle, batch)
            self.workspace = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            self.batch = batch

    def _check_inputs(self, mask_features, memories):
        want = torch.float32 if self.head.precision == 'fp32' else torch.bfloat16
        mf = mask_features.detach()
        if mf.dtype != want or not mf.is_contiguous():
            mf = mf.to(want).contiguous()
        mems = []
        for m in memories:
            m = m.detach()
            if m.dtype != want or not m.is_contiguous():
                m = m.to(want).contiguous()
            mems.append(m)
        return mf, mems

    # ---- whole path
    def forward(self, mask_features, memories, return_debug=False):
        h = self.head
        if h.cuda_graph and not return_debug:
            return self._forward_graph(mask_features, memories)
        return self._forward_eager(mask_features, memories, return_debug)

    def _forward_graph(self, mask_features, memories):
        """Replays a CUDA graph of the whole path.  ONE graph per (sizes, batch, weights): it is captured on the
        caller's input tensors the first time (kept alive with the graph) and replayed zero-copy as long as the
        caller keeps passing those same buffers; a call with other tensors of the same shape switches the entry to
        graph-owned static input buffers (one re-capture, then a device copy per call -- never a re-capture per
        step).  Any re-prepare (new sizes, batch or weights) drops the graphs, because they bake in the handle's
        tables and the workspace (see prepare()).  Outputs are graph-owned static tensors: the next replay
        overwrites them."""
        with torch.cuda.device(self.device):
            mf, mems = self._check_inputs(mask_features, memories)
            sizes = [tuple(m.shape[-2:]) for m in mems]
            self.prepare(mf.shape[2], mf.shape[3], sizes, mf.shape[0])       # may clear self._graphs
            key = (tuple(mf.shape), tuple(sizes), self.weights_key)
            ptrs = (mf.data_ptr(),) + tuple(m.data_ptr() for m in mems)
            entry = self._graphs.get(key)
            if entry is not None and entry['ptrs'] != ptrs:
                if not entry['owned']:
                    entry = None                                              # re-capture on graph-owned buffers
                    own = True
                else:
                    entry['mf'].copy_(mf)
                    for d, m in zip(entry['mems'], mems):
                        d.copy_(m)
            elif entry is None:
                own = False
            if entry is None:
                self._graphs.clear()
                if own:
                    mf, mems = mf.clone(), [m.clone() for m in mems]
                cur = torch.cuda.current_stream(self.device)
                side = torch.cuda.Stream(self.device, priority=-1)   # the layer chain outranks the helper streams
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    self._forward_eager(mf, mems, False)          # warm-up outside capture
                    side.synchronize()
                    g = torch.cuda.CUDAGraph()
                    with _lib.no_gc_during_capture(), torch.cuda.graph(g, stream=side):
                        outs = self._forward_eager(mf, mems, False)
                cur.wait_stream(side)
                entry = dict(graph=g, outs=outs, mf=mf, mems=mems, owned=own,
                             ptrs=(mf.data_ptr(),) + tuple(m.data_ptr() for m in mems) if own else ptrs)
                self._graphs[key] = entry
            entry['graph'].replay()
            return entry['outs']

    def _forward_eager(self, mask_features, memories, return_debug=False):
        h = self.head
        with torch.cuda.device(self.device):
            mf, mems = self._check_inputs(mask_features, memories)
            B, Cc, H4, W4 = mf.shape
            assert Cc == h.feat_channels and len(mems) == 3
            sizes = [tuple(m.shape[-2:]) for m in mems]
            self.prepare(H4, W4, sizes, B)
            L, Q = h.num_transformer_decoder_layers, h.num_queries
            dev = self.device
            cls = torch.empty((L + 1, B, Q, h.num_classes + 1), dtype=torch.float32, device=dev)
            emb = torch.empty((L + 1, B, Q, self.d_lang), dtype=torch.float32, device=dev) if self.d_lang else None
            n_maps = 1 if (h.final_mask_only and not return_debug) else L + 1
            mask = torch.empty((n_maps, B, Q, H4, W4), dtype=mf.dtype, device=dev)
            _lib.check(self.lib.cgg_set_final_mask_only(self.handle, int(n_maps == 1)), self.handle,
                       'cgg_set_final_mask_only')
            mem_ptrs = (C.c_void_p * 3)(*[m.data_ptr() for m in mems])
            xs = bms = am = None
            xs_p, bm_p, am_p = None, None, None
            if return_debug:
                xs = torch.empty((L + 1, B, Q, Cc), dtype=torch.float32, device=dev)
                bms = [torch.zeros((B, Q, (s[0] * s[1] + 31) // 32), dtype=torch.int32, device=dev)
                       for s in (sizes[j % 3] for j in range(L))]
                am = torch.zeros((L, B, Q), dtype=torch.uint8, device=dev)
                xs_p, am_p = _ptr(xs), _ptr(am)
                bm_p = (C.c_void_p * L)(*[b.data_ptr() for b in bms])
            st = self.lib.cgg_decoder_forward(self.handle, C.byref(self.weights), B, _ptr(mf), mem_ptrs, _ptr(cls),
                                              _ptr(emb) if emb is not None else None, _ptr(mask), xs_p, bm_p, am_p,
                                              _ptr(self.workspace),
                                              self.workspace.numel(), self._stream())
            _lib.check(st, self.handle, 'cgg_decoder_forward')
        masks = list(mask.unbind(0)) if mask.shape[0] == L + 1 else [None] * L + [mask[0]]
        cls_list = list(cls.unbind(0))
        # use_class_emb=False: cls_emb_pred = cls_pred (head.py:739-744)
        outs = (cls_list, list(emb.unbind(0)) if emb is not None else cls_list, masks)
        if return_debug:
            return outs + (dict(x=xs, bitmaps=bms, all_masked=am),)
        return outs

    def sine_pos(self, h, w):
        """(h*w, C) sine positional encoding (head.py:798-804), cached per size."""
        key = (h, w)
        if key not in self._pos:
            out = torch.empty((h * w, self.head.feat_channels), dtype=torch.float32, device=self.device)
            with torch.cuda.device(self.device):
                _lib.check(self.lib.cgg_sine_pos(self.handle, _ptr(out), h, w, self.head.feat_channels, self._stream()),
                           self.handle, 'cgg_sine_pos')
            self._pos[key] = out
        return self._pos[key]

    # ---- stages (parity tests, teacher forcing)
    def kv_project(self, memories):
        mem_ptrs = (C.c_void_p * 3)(*[m.data_ptr() for m in memories])
        _lib.check(self.lib.cgg_kv_project(self.handle, C.byref(self.weights), self.batch, mem_ptrs,
                                           _ptr(self.workspace), self.workspace.numel(), self._stream()),
                   self.handle, 'cgg_kv_project')

    def head_call(self, x, mask_features, target_level, want_bits=True):
        h = self.head
        B, Q = x.shape[0], h.num_queries
        H4, W4, sizes = self.sizes
        dev = self.device
        cls = torch.empty((B, Q, h.num_classes + 1), dtype=torch.float32, device=dev)
        emb = torch.empty((B, Q, self.d_lang), dtype=torch.float32, device=dev) if self.d_lang else None
        mask = torch.empty((B, Q, H4, W4), dtype=mask_features.dtype, device=dev)
        me = torch.empty((B, Q, h.feat_channels), dtype=torch.float32, device=dev)
        K = sizes[target_level][0] * sizes[target_level][1]
        bm = torch.zeros((B, Q, (K + 31) // 32), dtype=torch.int32, device=dev) if want_bits else None
        am = torch.zeros((B, Q), dtype=torch.uint8, device=dev) if want_bits else None
        st = self.lib.cgg_head_call(self.handle, C.byref(self.weights), B, _ptr(x), _ptr(mask_features), target_level,
                                    _ptr(cls), _ptr(emb) if emb is not None else None, _ptr(mask), _ptr(me),
                                    _ptr(bm) if want_bits else None,
                                    _ptr(am) if want_bits else None, _ptr(self.workspace), self.workspace.numel(),
                                    self._stream())
        _lib.check(st, self.handle, 'cgg_head_call')
        return cls, (emb if emb is not None else cls), mask, me, bm, am

    def mask_einsum(self, mask_features, mask_out, first_call=0, num_calls=None):
        """K2 alone (bf16 mode) from the mask embeddings already in the workspace; mask_out
        (num_calls, B, Q, H4, W4) bf16."""
        n = num_calls if num_calls is not None else mask_out.shape[0]
        st = self.lib.cgg_mask_einsum(self.handle, self.batch, first_call, n, _ptr(mask_features), _ptr(mask_out),
                                      _ptr(self.workspace), self.workspace.numel(), self._stream())
        _lib.check(st, self.handle, 'cgg_mask_einsum')

    def decoder_layer(self, layer, x, bitmap, all_masked):
        out = torch.empty_like(x)
        st = self.lib.cgg_decoder_layer(self.handle, C.byref(self.weights), x.shape[0], layer, _ptr(x),
                                        _ptr(bitmap) if bitmap is not None else None,
                                        _ptr(all_masked) if all_masked is not None else None, _ptr(out),
                                        _ptr(self.workspace), self.workspace.numel(), self._stream())
        _lib.check(st, self.handle, 'cgg_decoder_layer')
        return out

    def attn_mask_from_logits(self, mask_pred, target_hw):
        B, Q, H4, W4 = mask_pred.shape
        assert Q == self.head.num_queries and mask_pred.dtype == torch.float32 and mask_pred.is_contiguous()
        K = target_hw[0] * target_hw[1]
        bm = torch.zeros((B, Q, (K + 31) // 32), dtype=torch.int32, device=self.device)
        am = torch.zeros((B, Q), dtype=torch.uint8, device=self.device)
        st = self.lib.cgg_attn_mask_from_logits(self.handle, B, _ptr(mask_pred), H4, W4, target_hw[0], target_hw[1],
                                                _ptr(bm), _ptr(am), self._stream())
        _lib.check(st, self.handle, 'cgg_attn_mask_from_logits')
        return bm, am

    def masked_attention(self, q, k, v, bitmap=None, all_masked=None, layer=-1, out_half=False):
        """q (B,Q,C) pre-scaled fp32; k, v (B,K,C) views with unit channel stride and the same strides (fp32 in fp32
        mode, bf16 in bf16 mode), e.g. column slices of one K/V buffer.  layer >= 0 (bf16 mode): add decoder layer
        `layer`'s key-bias table to the keys, as that layer's cross-attention does.  Returns the fp32 output, or
        (fp32, IEEE half) outputs of the same launch with out_half=True."""
        B, Q, Cc = q.shape
        K = k.shape[1]
        assert k.stride() == v.stride() and k.stride(-1) == 1 and k.shape == v.shape, (k.stride(), v.stride())
        out = torch.empty_like(q)
        half = torch.empty(q.shape, dtype=torch.float16, device=q.device) if out_half else None
        st = self.lib.cgg_masked_attention(self.handle, B, K, _ptr(q), _ptr(k), _ptr(v), k.stride(1), k.stride(0),
                                           _ptr(bitmap) if bitmap is not None else None,
                                           _ptr(all_masked) if all_masked is not None else None, layer, _ptr(out),
                                           _ptr(half) if out_half else None, self._stream())
        _lib.check(st, self.handle, 'cgg_masked_attention')
        return (out, half) if out_half else out

    # ---- grounding side
    def similarity(self, a, b, scale):
        a = a.detach().float().contiguous()
        b = b.detach().float().contiguous()
        out = torch.empty((a.shape[0], b.shape[0]), dtype=torch.float32, device=self.device)
        st = self.lib.cgg_similarity(self.handle, _ptr(a), _ptr(b), a.shape[0], b.shape[0], a.shape[1], scale,
                                     _ptr(out), self._stream())
        _lib.check(st, self.handle, 'cgg_similarity')
        return out

    def noun_embeddings(self, table, ln_w, ln_b, ids, eps, text_emb_norm):
        ids = ids.contiguous()
        out = torch.empty(tuple(ids.shape) + (table.shape[1],), dtype=torch.float32, device=self.device)
        st = self.lib.cgg_noun_embeddings(self.handle, _ptr(table), _ptr(ln_w), _ptr(ln_b), _ptr(ids), ids.numel(),
                                          table.shape[1], eps, int(bool(text_emb_norm)), _ptr(out), self._stream())
        _lib.check(st, self.handle, 'cgg_noun_embeddings')
        return out

    def grounding_loss(self, pred, cap, cap_mask, temperature, loss_weight):
        pred, cap = pred.detach().float().contiguous(), cap.detach().float().contiguous()
        cap_mask = cap_mask.to(torch.int64).contiguous()
        Bg, Q, D = pred.shape
        T = cap.shape[1]
        nbytes = self.lib.cgg_grounding_scratch_bytes(Bg, Q, T)
        scratch = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        loss = torch.empty(1, dtype=torch.float32, device=self.device)
        st = self.lib.cgg_grounding_loss(self.handle, _ptr(pred), _ptr(cap), _ptr(cap_mask), Bg, Q, T, D, temperature,
                                         loss_weight, _ptr(loss), _ptr(scratch), nbytes, self._stream())
        _lib.check(st, self.handle, 'cgg_grounding_loss')
        return loss[0]


def build_head_from_state_dict(sd, num_queries, num_classes_p1=49, precision='fp32', device='cuda', num_layers=9,
                               cuda_graph=False, final_mask_only=False, num_stuff_classes=0, **kwargs):
    """Convenience used by tests / bench: a head carrying the given (reference-keyed) weights.  The last
    num_stuff_classes of the num_classes_p1 - 1 classes are stuff (panoptic output), the others things."""
    kwargs.setdefault('use_class_emb', 'v2l_transform.weight' in sd)
    head = Mask2FormerHeadOpenB200(num_things_classes=num_classes_p1 - 1 - num_stuff_classes,
                                   num_stuff_classes=num_stuff_classes,
                                   num_queries=num_queries, precision=precision, cuda_graph=cuda_graph,
                                   final_mask_only=final_mask_only, **kwargs,
                                   transformer_decoder=dict(num_layers=num_layers))
    missing = head.load_state_dict(sd, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    return head.to(device).eval()
