"""ctypes binding of the C-ABI library (include/cgg_b200.h).  There is no fallback: if
libcgg_b200.so is missing or a call fails, this raises."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('CGG_LIB', os.path.join(HERE, 'libcgg_b200.so'))   # CGG_LIB: A/B another build of the same ABI

MAX_LAYERS = 16
NUM_LEVELS = 3
FP32, BF16 = 0, 1
c_float_p = C.POINTER(C.c_float)

EXPORTS = ['cgg_create', 'cgg_destroy', 'cgg_last_error', 'cgg_version', 'cgg_launch_count', 'cgg_prepare', 'cgg_workspace_bytes', 'cgg_workspace_offset',
           'cgg_decoder_forward', 'cgg_kv_project', 'cgg_head_call', 'cgg_attn_mask_from_logits',
           'cgg_decoder_layer', 'cgg_mask_einsum', 'cgg_masked_attention', 'cgg_noun_embeddings', 'cgg_similarity',
           'cgg_grounding_scratch_bytes', 'cgg_grounding_loss', 'cgg_grounding_bwd_scratch_bytes',
           'cgg_grounding_loss_backward', 'cgg_set_final_mask_only',
           # training-step stages
           'cgg_gemm_f32', 'cgg_layernorm', 'cgg_layernorm_bwd_scratch_bytes', 'cgg_layernorm_backward', 'cgg_relu_backward',
           'cgg_axpy', 'cgg_add_rows', 'cgg_sum_batch', 'cgg_colsum', 'cgg_mem_prep', 'cgg_mem_prep_backward', 'cgg_sine_pos',
           'cgg_attention_f32', 'cgg_attention_backward', 'cgg_attn_softmax_rows', 'cgg_attn_dscore', 'cgg_point_sample', 'cgg_point_sample_backward',
           'cgg_matching_cost', 'cgg_panoptic_stuff_labels', 'cgg_gt_point_sample', 'cgg_point_losses', 'cgg_point_losses_backward', 'cgg_weighted_ce', 'cgg_weighted_ce_backward',
           # test-time step after the path
           'cgg_upsample_masks', 'cgg_instance_mask_stats', 'cgg_softmax_rows', 'cgg_panoptic_scratch_bytes',
           'cgg_panoptic_fuse', 'cgg_caption_self_attn_step', 'cgg_caption_cache_reorder', 'cgg_caption_beam_scores',
           'cgg_caption_beam_select',
           # the pixel decoder before the path
           'cgg_ms_deform_attn', 'cgg_ms_deform_attn_backward', 'cgg_group_norm_scratch_bytes', 'cgg_group_norm_tokens',
           'cgg_group_norm_tokens_backward', 'cgg_upsample_add_tokens', 'cgg_upsample_add_tokens_backward',
           'cgg_tokens_to_nchw', 'cgg_nchw_to_tokens']


class Config(C.Structure):
    _fields_ = [(n, C.c_int) for n in ('num_queries', 'embed_dim', 'num_heads', 'ffn_dim', 'num_layers',
                                       'num_classes_p1', 'd_lang', 'precision', 'pred_emb_norm')]


class LayerWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ('cross_in_w', 'cross_in_b', 'cross_out_w', 'cross_out_b', 'self_in_w',
                                          'self_in_b', 'self_out_w', 'self_out_b', 'ffn_w1', 'ffn_b1', 'ffn_w2',
                                          'ffn_b2')] + [('norm_w', C.c_void_p * 3), ('norm_b', C.c_void_p * 3)]


class Weights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ('query_embed', 'query_feat', 'level_embed', 'cls_w', 'cls_b')] + \
               [('me_w', C.c_void_p * 3), ('me_b', C.c_void_p * 3)] + \
               [(n, C.c_void_p) for n in ('v2l_w', 'v2l_b', 'post_norm_w', 'post_norm_b')] + \
               [('layers', LayerWeights * MAX_LAYERS)]


class GemmDesc(C.Structure):
    """cgg_gemm_desc (include/cgg_b200.h)"""
    _fields_ = [('A', C.c_void_p), ('sAb', C.c_long), ('sAm', C.c_long), ('sAk', C.c_long),
                ('A2', C.c_void_p), ('sA2m', C.c_long), ('sA2k', C.c_long), ('a2_mod', C.c_int),
                ('W', C.c_void_p), ('sWb', C.c_long), ('sWn', C.c_long), ('sWk', C.c_long),
                ('bias', C.c_void_p),
                ('R', C.c_void_p), ('sRb', C.c_long), ('sRm', C.c_long), ('sRn', C.c_long), ('r_mod', C.c_int),
                ('r_ncols', C.c_int),
                ('C', C.c_void_p), ('sCb', C.c_long), ('sCm', C.c_long), ('sCn', C.c_long),
                ('M', C.c_int), ('N', C.c_int), ('K', C.c_int), ('batch', C.c_int),
                ('relu', C.c_int), ('alpha', C.c_float), ('a_mmajor', C.c_int), ('c_mmajor', C.c_int), ('tf32', C.c_int),
                ('batch_inner', C.c_int), ('sAb2', C.c_long), ('sWb2', C.c_long), ('sCb2', C.c_long), ('accumulate', C.c_int), ('slot', C.c_int), ('conv_cin', C.c_int)]


class BeamState(C.Structure):
    """cgg_beam_state (include/cgg_b200.h): device pointers of a batched caption beam search"""
    _fields_ = [('tokens', C.c_void_p), ('token_cap', C.c_int)] + \
               [(n, C.c_void_p) for n in ('weights', 'n_active', 'parent', 'next_ids', 'fin_tokens', 'fin_len', 'fin_score',
                                         'n_fin', 'max_idx', 'done', 'n_done')]


class GtImage(C.Structure):
    """cgg_gt_image (include/cgg_b200.h): one image's compact panoptic training targets (device pointers)"""
    _fields_ = [('things', C.c_void_p), ('sem', C.c_void_p), ('stuff_labels', C.c_void_p), ('sem_stride', C.c_int64)] + \
               [(n, C.c_int) for n in ('num_things', 'h', 'w', 'pad_h', 'pad_w', 'num_stuff', 'sem_is_i64', 'reserved')]


class CggError(RuntimeError):
    pass


_lib = None


def load():
    """Loads the shared library; raises if it has not been built (no CPU / torch fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CggError('%s not found: build it with `python -m cgg_b200.build` '
                       '(there is no fallback path)' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp, i, sz = C.c_void_p, C.c_int, C.c_size_t
    lib.cgg_create.argtypes = [C.POINTER(vp), C.POINTER(Config)]
    lib.cgg_destroy.argtypes = [vp]
    lib.cgg_destroy.restype = None
    lib.cgg_last_error.argtypes = [vp]
    lib.cgg_last_error.restype = C.c_char_p
    lib.cgg_version.restype = C.c_char_p
    lib.cgg_launch_count.restype = C.c_uint64
    lib.cgg_prepare.argtypes = [vp, C.POINTER(Weights), i, i, C.POINTER(i), C.POINTER(i), vp]
    lib.cgg_workspace_bytes.argtypes = [vp, i]
    lib.cgg_workspace_bytes.restype = sz
    lib.cgg_workspace_offset.argtypes = [vp, i, C.c_char_p]
    lib.cgg_workspace_offset.restype = sz
    lib.cgg_decoder_forward.argtypes = [vp, C.POINTER(Weights), i, vp, C.POINTER(vp), vp, vp, vp, vp,
                                        C.POINTER(vp), vp, vp, sz, vp]
    lib.cgg_kv_project.argtypes = [vp, C.POINTER(Weights), i, C.POINTER(vp), vp, sz, vp]
    lib.cgg_head_call.argtypes = [vp, C.POINTER(Weights), i, vp, vp, i, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    lib.cgg_mask_einsum.argtypes = [vp, i, i, i, vp, vp, vp, sz, vp]
    lib.cgg_attn_mask_from_logits.argtypes = [vp, i, vp, i, i, i, i, vp, vp, vp]
    lib.cgg_decoder_layer.argtypes = [vp, C.POINTER(Weights), i, i, vp, vp, vp, vp, vp, sz, vp]
    lib.cgg_masked_attention.argtypes = [vp, i, i, vp, vp, vp, C.c_long, C.c_long, vp, vp, i, vp, vp, vp]
    lib.cgg_noun_embeddings.argtypes = [vp, vp, vp, vp, vp, i, i, C.c_float, i, vp, vp]
    lib.cgg_similarity.argtypes = [vp, vp, vp, i, i, i, C.c_float, vp, vp]
    lib.cgg_grounding_scratch_bytes.argtypes = [i, i, i]
    lib.cgg_grounding_scratch_bytes.restype = sz
    lib.cgg_grounding_loss.argtypes = [vp, vp, vp, vp, i, i, i, i, C.c_float, C.c_float, vp, vp, sz, vp]
    lib.cgg_set_final_mask_only.argtypes = [vp, i]
    lib.cgg_grounding_bwd_scratch_bytes.argtypes = [i, i, i]
    lib.cgg_grounding_bwd_scratch_bytes.restype = sz
    lib.cgg_grounding_loss_backward.argtypes = [vp, vp, vp, vp, i, i, i, i, C.c_float, C.c_float, C.c_float, vp, vp, sz, vp]
    f32, lg = C.c_float, C.c_long
    lib.cgg_gemm_f32.argtypes = [vp, C.POINTER(GemmDesc), vp]
    lib.cgg_layernorm.argtypes = [vp, vp, vp, vp, vp, i, i, f32, vp]
    lib.cgg_layernorm_bwd_scratch_bytes.argtypes = [i, i]
    lib.cgg_layernorm_bwd_scratch_bytes.restype = sz
    lib.cgg_layernorm_backward.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, sz, i, i, f32, vp]
    lib.cgg_relu_backward.argtypes = [vp, vp, vp, vp, lg, f32, vp]
    lib.cgg_axpy.argtypes = [vp, vp, vp, lg, f32, vp]
    lib.cgg_add_rows.argtypes = [vp, vp, vp, vp, i, lg, vp]
    lib.cgg_sum_batch.argtypes = [vp, vp, vp, i, lg, vp]
    lib.cgg_colsum.argtypes = [vp, vp, vp, lg, i, f32, i, vp]
    lib.cgg_mem_prep.argtypes = [vp, vp, vp, vp, vp, vp, i, i, i, vp]
    lib.cgg_mem_prep_backward.argtypes = [vp, vp, vp, vp, i, i, i, vp]
    lib.cgg_sine_pos.argtypes = [vp, vp, i, i, i, vp]
    lib.cgg_attention_f32.argtypes = [vp, i, i, i, i, vp, vp, vp, lg, lg, vp, vp, vp, vp]
    lib.cgg_attention_backward.argtypes = [vp, i, i, i, i, vp, vp, vp, lg, lg, vp, vp, vp, vp, vp, vp, vp, lg, lg, vp, vp]
    lib.cgg_attn_softmax_rows.argtypes = [vp, vp, vp, vp, i, i, i, i, vp]
    lib.cgg_attn_dscore.argtypes = [vp, vp, vp, vp, vp, i, i, i, i, i, vp]
    f = C.c_float
    lib.cgg_point_sample.argtypes = [vp, vp, vp, vp, i, i, i, i, i, vp]
    lib.cgg_point_sample_backward.argtypes = [vp, vp, vp, vp, i, i, i, i, i, vp]
    lib.cgg_matching_cost.argtypes = [vp, vp, vp, vp, vp, vp, i, i, i, i, f, f, f, f, f, vp, vp, vp]
    lib.cgg_panoptic_stuff_labels.argtypes = [vp, vp, i, i, i, i, i, i, vp, vp, vp, vp]
    lib.cgg_gt_point_sample.argtypes = [vp, vp, vp, vp, vp, i, i, i, vp]
    lib.cgg_point_losses.argtypes = [vp, vp, vp, i, i, f, vp, vp, vp, vp]
    lib.cgg_point_losses_backward.argtypes = [vp, vp, vp, vp, i, i, f, vp, vp, vp, vp]
    lib.cgg_weighted_ce.argtypes = [vp, vp, vp, vp, i, i, vp, vp, vp, vp]
    lib.cgg_weighted_ce_backward.argtypes = [vp, vp, vp, vp, vp, i, i, vp, vp, vp]
    lib.cgg_upsample_masks.argtypes = [vp, vp, i, vp, i, i, i, i, i, vp]
    lib.cgg_instance_mask_stats.argtypes = [vp, vp, i, vp, i, i, i, i, i, i, i, i, vp, vp, vp, vp, vp]
    lib.cgg_softmax_rows.argtypes = [vp, vp, i, i, vp]
    lib.cgg_panoptic_scratch_bytes.argtypes = [i, i]
    lib.cgg_panoptic_scratch_bytes.restype = sz
    dbl = C.c_double
    lib.cgg_panoptic_fuse.argtypes = [vp, vp, i, vp, vp, i, i, i, i, i, i, i, i, i, i, dbl, dbl, i, vp, vp, vp, vp, vp, sz, vp]
    bs = C.POINTER(BeamState)
    lib.cgg_caption_self_attn_step.argtypes = [vp, vp, vp, vp, vp, i, i, i, i, i, f32, vp]
    lib.cgg_caption_cache_reorder.argtypes = [vp, vp, vp, vp, i, i, i, i, i, i, vp]
    lib.cgg_caption_beam_scores.argtypes = [vp, vp, i, i, i, i, i, bs, f32, vp, vp, vp]
    lib.cgg_caption_beam_select.argtypes = [vp, vp, vp, i, i, i, i, i, i, f32, f32, i, bs, vp]
    ip = C.POINTER(C.c_int)
    lib.cgg_ms_deform_attn.argtypes = [vp, vp, lg, vp, lg, vp, lg, vp, i, i, i, i, i, ip, ip, vp]
    lib.cgg_ms_deform_attn_backward.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i, i, i, i, i, ip, ip, vp]
    lib.cgg_group_norm_scratch_bytes.argtypes = [i, i, i, i]
    lib.cgg_group_norm_scratch_bytes.restype = sz
    lib.cgg_group_norm_tokens.argtypes = [vp, vp, vp, vp, vp, vp, vp, sz, i, i, i, i, f32, i, vp]
    lib.cgg_group_norm_tokens_backward.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, i, i, i, i, vp]
    lib.cgg_upsample_add_tokens.argtypes = [vp, vp, vp, lg, vp, i, i, i, i, i, i, vp]
    lib.cgg_upsample_add_tokens_backward.argtypes = [vp, vp, vp, i, i, i, i, i, i, vp]
    lib.cgg_tokens_to_nchw.argtypes = [vp, vp, lg, vp, i, i, i, i, vp]
    lib.cgg_nchw_to_tokens.argtypes = [vp, vp, vp, lg, i, i, i, i, vp]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if fn.restype is C.c_int and name not in ('cgg_destroy',):
            fn.restype = C.c_int
    _lib = lib
    return lib


STATUS = {0: 'CGG_OK', -1: 'CGG_ERR_BAD_SHAPE', -2: 'CGG_ERR_UNSUPPORTED', -3: 'CGG_ERR_CUDA',
          -4: 'CGG_ERR_NOT_PREPARED', -5: 'CGG_ERR_WORKSPACE', -6: 'CGG_ERR_NULL'}


def check(status, handle=None, what=''):
    if status != 0:
        msg = ''
        if handle:
            msg = load().cgg_last_error(handle).decode()
        raise CggError('%s failed: %s %s' % (what, STATUS.get(status, status), msg))


class no_gc_during_capture:
    """Context for a CUDA-graph capture: collects garbage first and keeps the cyclic collector off while the stream is
    capturing.  A head and its runtime reference each other, so a dropped head is freed by the CYCLIC collector, at an
    arbitrary later allocation -- and its `cgg_destroy` (cudaFree, cudaStreamDestroy) in the middle of a global-mode capture
    invalidates the capture (cudaErrorStreamCaptureInvalidated at the next launch).  torch.cuda.graph no longer collects on
    entry by itself."""

    def __enter__(self):
        import gc
        self._was = gc.isenabled()
        gc.collect()
        gc.disable()
        return self

    def __exit__(self, *exc):
        import gc
        if self._was:
            gc.enable()
        return False

