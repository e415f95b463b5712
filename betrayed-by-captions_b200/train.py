"""Training step of the decoder head: the forward of `Mask2FormerHeadOpen.forward` (mask2former_head.py:763-849) as an
autograd graph whose every node is a kernel of the C-ABI library -- forward AND backward -- so that
`forward_train -> loss -> backward` (mask2former_head.py:851-921, :393-462) reaches every parameter of the head, the
pixel-decoder features and the memories exactly as the reference's autograd does (SURVEY.md App. B item 12: the
attention mask is detached, nothing flows through K3).

PyTorch is the tape (autograd.Function), the allocator and the stream; it computes nothing here.  With
`train_precision='fp32'` all arithmetic is fp32 FMA (the parity mode extended with gradients); with 'tf32' every
contraction -- each linear layer, the mask einsum and all of their dX / dW products -- runs on tcgen05 kind::tf32 MMAs
fed by TMA from the same fp32 tensors (csrc/gemm_tf32.cu), everything else stays fp32.  Gradient all-reduce over NVLink for data-parallel
training lives in `GradReducer` below (bucketed NCCL all-reduce overlapped with the backward; reference: mmcv's
MMDistributedDataParallel built at open_set/apis/train.py:156-161).
"""
import ctypes as C
import math

import torch
import torch.distributed as dist

from . import lib as _lib


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


class _K:
    """Thin launcher over the stage entry points of include/cgg_b200.h for one runtime (handle + device)."""

    def __init__(self, rt, tf32=False):
        self.rt, self.lib, self.h, self.dev = rt, rt.lib, rt.handle, rt.device
        self.tf32 = int(bool(tf32))      # contractions on tcgen05 kind::tf32 MMAs instead of fp32 FMAs
        self.slot = 0
        self.wgrad = None                # _WgradSide of the step being recorded (fused weight gradients), or None

    def s(self):
        return C.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)

    def chk(self, st, what):
        _lib.check(st, self.h, what)

    def new(self, *shape):
        return torch.empty(shape, dtype=torch.float32, device=self.dev)

    def gemm(self, A, sA, W, sW, Cc, sC, M, N, K, batch=1, bias=None, R=None, sR=(0, 0, 0), r_mod=None, alpha=1.0,
             relu=False, a_mmajor=False, c_mmajor=False, batch_inner=1, s2=(0, 0, 0), accumulate=False, conv_cin=0, r_ncols=1 << 30):
        """C[b,m,n] = relu?((sum_k A[b,m,k] W[b,n,k] + bias[n]) * alpha + R[b, m % r_mod, n]); element strides
        sA = (b, m, k), sW = (b, n, k), sC = (b, m, n), sR = (b, m, n)."""
        d = _lib.GemmDesc()
        d.A, (d.sAb, d.sAm, d.sAk) = A.data_ptr(), sA
        d.A2, d.a2_mod = None, 1
        d.W, (d.sWb, d.sWn, d.sWk) = W.data_ptr(), sW
        d.bias = bias.data_ptr() if bias is not None else None
        if R is not None:
            d.R, (d.sRb, d.sRm, d.sRn) = R.data_ptr(), sR
            d.r_mod = r_mod if r_mod is not None else M
        else:
            d.R, d.r_mod = None, 1
        d.r_ncols = r_ncols                                           # the residual applies to columns n < r_ncols
        d.C, (d.sCb, d.sCm, d.sCn) = Cc.data_ptr(), sC
        d.M, d.N, d.K, d.batch = M, N, K, batch
        d.relu, d.alpha = int(relu), float(alpha)
        d.a_mmajor, d.c_mmajor = int(a_mmajor), int(c_mmajor)
        d.tf32 = self.tf32
        d.batch_inner, (d.sAb2, d.sWb2, d.sCb2) = batch_inner, s2     # (image, head) batches: inner strides of A, W, C
        d.accumulate = int(accumulate)                                # C += result (in-place gradient accumulation)
        d.slot = self.slot                                            # split-K workspace (1 on the weight-gradient side stream)
        d.conv_cin = conv_cin                                         # 3x3 convolution as an implicit GEMM (pixel decoder)
        self.chk(self.lib.cgg_gemm_f32(self.h, C.byref(d), self.s()), 'cgg_gemm_f32')


# ------------------------------------------------------------------------------------------- autograd nodes
class _WgradSide:
    """Weight / bias gradients of the linear layers written straight into the parameters' `.grad` (the GradReducer's
    bucket views, or any pre-allocated .grad) by the GEMM epilogue (`accumulate`), on a SIDE stream: they are leaves of the
    backward, so the dX chain on the main stream never waits for them, and autograd's own accumulation kernels
    (`p.grad += dW`, the slice scatter of the fused in-projections) disappear.  Autograd gets None for these gradients;
    the reducer (if any) is told directly when a parameter's gradient is complete.  The side stream joins the main stream
    in an engine callback at the end of the backward."""

    _side = {}

    def __init__(self, dev):
        if dev not in _WgradSide._side:
            _WgradSide._side[dev] = torch.cuda.Stream(dev)
        self.dev, self.stream = dev, _WgradSide._side[dev]
        self.parts = {}          # parameter -> number of fused products that write into its .grad
        self.done = {}
        self.queued = False
        self.keep = []           # operands of the side-stream products: alive until the join (no allocator reuse under them)

    def target(self, param, view):
        """Registers `view` (param.grad or a slice of it) as the destination of one fused product; None if not possible."""
        if view is None:
            return None
        self.parts[param] = self.parts.get(param, 0) + 1
        return (param, view)

    def launch(self, k, fn, keep):
        """Runs fn() (kernel launches) on the side stream after everything issued so far on the current stream.  Outside
        a graph capture the products are issued in line instead: the fork / join events would cost the host more than the
        overlap gives a launch-bound eager step (the in-place accumulation is what matters there)."""
        if not torch.cuda.is_current_stream_capturing():
            self.inline = True
            slot, k.slot = k.slot, 1       # (the side stream's split-K workspace: sized here, before any capture)
            try:
                fn()
            finally:
                k.slot = slot
            return
        self.inline = False
        main = torch.cuda.current_stream(self.dev)
        ev = torch.cuda.Event()
        ev.record(main)
        self.stream.wait_event(ev)
        slot = k.slot
        with torch.cuda.stream(self.stream):
            k.slot = 1
            try:
                fn()
            finally:
                k.slot = slot
        self.keep.extend(keep)
        if not self.queued:
            self.queued = True
            torch.autograd.Variable._execution_engine.queue_callback(self.join)

    def written(self, param):
        self.done[param] = self.done.get(param, 0) + 1
        if self.done[param] == self.parts.get(param, 1):
            red = _FUSED_REDUCERS.get(param)
            if red is not None:
                red.param_done(param, None if getattr(self, 'inline', False) else self.stream)

    def join(self):
        torch.cuda.current_stream(self.dev).wait_stream(self.stream)
        self.queued = False
        self.done = {}
        self.keep = []


_FUSED_REDUCERS = {}        # parameter -> GradReducer that must hear about gradients written outside autograd


class _Linear(torch.autograd.Function):
    """y = relu?((x W^T + b) * alpha + res).  x (rows, K) contiguous, W (N, K), res (rows, N) or None.
    wdst / bdst: optional (parameter, grad view) pairs from _WgradSide.target: the weight / bias gradient is then
    accumulated into that view on the side stream and None is returned for it."""

    @staticmethod
    def forward(ctx, k, x, W, b, res, alpha, relu, wdst=None, bdst=None):
        rows, Kd = x.shape
        N = W.shape[0]
        y = k.new(rows, N)
        k.gemm(x, (0, Kd, 1), W, (0, Kd, 1), y, (0, N, 1), rows, N, Kd, bias=b, R=res, sR=(0, N, 1), r_mod=rows,
               alpha=alpha, relu=relu)
        ctx.k, ctx.alpha, ctx.relu, ctx.has_res, ctx.has_b = k, alpha, relu, res is not None, b is not None
        ctx.wdst, ctx.bdst, ctx.wgrad = wdst, bdst, k.wgrad
        ctx.save_for_backward(x, W, y if relu else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        k = ctx.k
        x, W, y = ctx.saved_tensors
        rows, Kd = x.shape
        N = W.shape[0]
        dy = dy.contiguous()
        g = dy
        if ctx.relu:                                      # (never combined with a residual on this path)
            g = k.new(rows, N)
            k.chk(k.lib.cgg_relu_backward(k.h, _p(y), _p(dy), _p(g), rows * N, 1.0, k.s()), 'cgg_relu_backward')
        dx = dW = db = None
        side = ctx.wgrad
        fuse_w = side is not None and ctx.wdst is not None and ctx.needs_input_grad[2]
        fuse_b = side is not None and ctx.bdst is not None and ctx.has_b and ctx.needs_input_grad[3]
        if fuse_w or fuse_b:
            def leaves():
                if fuse_w:                                # W.grad[n,kk] += alpha * sum_m g[m,n] x[m,kk]
                    k.gemm(g, (0, 1, N), x, (0, 1, Kd), ctx.wdst[1], (0, Kd, 1), N, Kd, rows, alpha=ctx.alpha, a_mmajor=True,
                           accumulate=True)
                if fuse_b:
                    k.chk(k.lib.cgg_colsum(k.h, _p(g), _p(ctx.bdst[1]), rows, N, ctx.alpha, 1, k.s()), 'cgg_colsum')
            side.launch(k, leaves, (g, x))
            if fuse_w:
                side.written(ctx.wdst[0])
            if fuse_b:
                side.written(ctx.bdst[0])
        if ctx.needs_input_grad[1]:                       # dx[m,kk] = alpha * sum_n g[m,n] W[n,kk]
            dx = k.new(rows, Kd)
            k.gemm(g, (0, N, 1), W, (0, 1, Kd), dx, (0, Kd, 1), rows, Kd, N, alpha=ctx.alpha)
        if ctx.needs_input_grad[2] and not fuse_w:        # dW[n,kk] = alpha * sum_m g[m,n] x[m,kk]
            dW = k.new(N, Kd)
            k.gemm(g, (0, 1, N), x, (0, 1, Kd), dW, (0, Kd, 1), N, Kd, rows, alpha=ctx.alpha, a_mmajor=True)
        if ctx.has_b and ctx.needs_input_grad[3] and not fuse_b:
            db = k.new(N)
            k.chk(k.lib.cgg_colsum(k.h, _p(g), _p(db), rows, N, ctx.alpha, 0, k.s()), 'cgg_colsum')
        dres = dy if (ctx.has_res and ctx.needs_input_grad[4]) else None
        if dres is not None and (fuse_w or fuse_b) and not getattr(side, 'inline', True):
            # autograd may add the residual stream's other gradients INTO the tensor it is handed, on the main stream,
            # while the side stream still reads dy: it gets its own copy
            dres = dy.clone()
        return None, dx, dW, db, dres, None, None, None, None


class _LayerNorm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, k, x, w, b, eps):
        rows, n = x.shape
        y = k.new(rows, n)
        k.chk(k.lib.cgg_layernorm(k.h, _p(x), _p(w), _p(b), _p(y), rows, n, eps, k.s()), 'cgg_layernorm')
        ctx.k, ctx.eps = k, eps
        ctx.save_for_backward(x, w)
        return y

    @staticmethod
    def backward(ctx, dy):
        k = ctx.k
        x, w = ctx.saved_tensors
        rows, n = x.shape
        dy = dy.contiguous()
        dx, dw, db = k.new(rows, n), k.new(n), k.new(n)
        nb = k.lib.cgg_layernorm_bwd_scratch_bytes(rows, n)
        scratch = torch.empty(nb, dtype=torch.uint8, device=k.dev)
        k.chk(k.lib.cgg_layernorm_backward(k.h, _p(x), _p(w), _p(dy), _p(dx), _p(dw), _p(db), _p(scratch), nb, rows, n,
                                           ctx.eps, k.s()), 'cgg_layernorm_backward')
        return None, dx, dw, db, None


class _AddRows(torch.autograd.Function):
    """out[b] = x[b] + add  (x (B, M, K) or None = zeros; add (M, K)): `x + query_embed`, the query_feat broadcast."""

    @staticmethod
    def forward(ctx, k, x, add, batch):
        per = add.numel()
        out = k.new(batch, *add.shape)
        k.chk(k.lib.cgg_add_rows(k.h, _p(x), _p(add), _p(out), batch, per, k.s()), 'cgg_add_rows')
        ctx.k, ctx.batch, ctx.has_x = k, batch, x is not None
        return out

    @staticmethod
    def backward(ctx, g):
        k = ctx.k
        g = g.contiguous()
        dadd = None
        if ctx.needs_input_grad[2]:
            dadd = k.new(*g.shape[1:])
            per = dadd.numel()
            if ctx.batch > per and (ctx.batch + 255) // 256 <= 65535:
                # many short rows (a level embedding added to every pixel's position row): a column sum over `batch` rows --
                # cgg_sum_batch would walk the whole batch with `per` threads
                k.chk(k.lib.cgg_colsum(k.h, _p(g), _p(dadd), ctx.batch, per, 1.0, 0, k.s()), 'cgg_colsum')
            else:
                k.chk(k.lib.cgg_sum_batch(k.h, _p(g), _p(dadd), ctx.batch, per, k.s()), 'cgg_sum_batch')
        return None, (g if ctx.has_x else None), dadd, None


class _MemPrep(torch.autograd.Function):
    """key_in = mem^T + level + pos, val_in = mem^T + level (head.py:792-804); mem (B, C, h, w) -> (B, K, C) x 2."""

    @staticmethod
    def forward(ctx, k, mem, level, pos):
        B, Cc, h, w = mem.shape
        K = h * w
        pos_level = k.new(K, Cc)
        k.chk(k.lib.cgg_add_rows(k.h, _p(pos), _p(level), _p(pos_level), K, Cc, k.s()), 'cgg_add_rows')   # pos + level
        key_in, val_in = k.new(B, K, Cc), k.new(B, K, Cc)
        k.chk(k.lib.cgg_mem_prep(k.h, _p(mem), _p(level), _p(pos_level), _p(key_in), _p(val_in), B, Cc, K, k.s()),
              'cgg_mem_prep')
        ctx.k, ctx.shape = k, (B, Cc, h, w)
        return key_in, val_in

    @staticmethod
    def backward(ctx, dkey, dval):
        k = ctx.k
        B, Cc, h, w = ctx.shape
        K = h * w
        dkey, dval = dkey.contiguous(), dval.contiguous()
        dmem = dlevel = None
        if ctx.needs_input_grad[1]:
            dmem = k.new(B, Cc, h, w)
            k.chk(k.lib.cgg_mem_prep_backward(k.h, _p(dkey), _p(dval), _p(dmem), B, Cc, K, k.s()), 'cgg_mem_prep_backward')
        if ctx.needs_input_grad[2]:
            a, b2 = k.new(Cc), k.new(Cc)
            k.chk(k.lib.cgg_colsum(k.h, _p(dkey), _p(a), B * K, Cc, 1.0, 0, k.s()), 'cgg_colsum')
            k.chk(k.lib.cgg_colsum(k.h, _p(dval), _p(b2), B * K, Cc, 1.0, 0, k.s()), 'cgg_colsum')
            k.chk(k.lib.cgg_axpy(k.h, _p(b2), _p(a), Cc, 1.0, k.s()), 'cgg_axpy')
            dlevel = a
        return None, dmem, dlevel, None


class _Attention(torch.autograd.Function):
    """softmax(q k^T + mask) v over `heads` heads of 32 channels, the flash-style fp32 kernels.  q (B, Q, C) scaled;
    k, v (B, K, C); bitmap / all_masked or None."""

    @staticmethod
    def forward(ctx, k_, q, kk, v, bitmap, all_masked, heads):
        B, Q, Cc = q.shape
        K = kk.shape[1]
        out = k_.new(B, Q, Cc)
        k_.chk(k_.lib.cgg_attention_f32(k_.h, B, Q, K, heads, _p(q), _p(kk), _p(v), Cc, K * Cc, _p(bitmap), _p(all_masked),
                                        _p(out), k_.s()), 'cgg_attention_f32')
        ctx.k, ctx.heads = k_, heads
        ctx.save_for_backward(q, kk, v, out, bitmap, all_masked)
        return out

    @staticmethod
    def backward(ctx, dout):
        k_, heads = ctx.k, ctx.heads
        q, kk, v, out, bitmap, all_masked = ctx.saved_tensors
        B, Q, Cc = q.shape
        K = kk.shape[1]
        dout = dout.contiguous()
        dq, dk, dv = k_.new(B, Q, Cc), k_.new(B, K, Cc), k_.new(B, K, Cc)
        scratch = k_.new(2 * B * heads * Q)
        k_.chk(k_.lib.cgg_attention_backward(k_.h, B, Q, K, heads, _p(q), _p(kk), _p(v), Cc, K * Cc, _p(bitmap),
                                             _p(all_masked), _p(out), _p(dout), _p(dq), _p(dk), _p(dv), Cc, K * Cc,
                                             _p(scratch), k_.s()), 'cgg_attention_backward')
        return None, dq, dk, dv, None, None, None


class _AttentionViews(torch.autograd.Function):
    """softmax(scale * q k^T | bitmap) v as tensor-core products, the GEMM-form attention of the decoder's tf32 training
    mode and of the caption transformer (row f4: 8 heads x 96).  q4, k4, v4 are (B, L, H, d) VIEWS (last stride 1, any
    row / head / batch strides: e.g. the three slices of a fused qkv projection) -> (B, Lq, H*d) contiguous.
    S = q k^T, P = softmax(S | bitmap), O = P v and the four gradient products are calls of the tcgen05 GEMM over
    (image, head) batches; P is kept for the backward (B * H * Lq * Lk floats).  A bit set in bitmap (B, Lq, ceil(Lk/32))
    excludes the key; an all_masked row attends every key; a row with no key left gives zeros."""

    @staticmethod
    def forward(ctx, k_, q4, k4, v4, bitmap, all_masked, scale):
        B, Lq, H, d = q4.shape
        Lk = k4.shape[1]
        for t in (q4, k4, v4):
            assert t.stride(3) == 1 and t.dtype == torch.float32
        P = k_.new(B, H, Lq, Lk)
        bh = dict(batch=B * H, batch_inner=H)
        sq, sk, sv = q4.stride(), k4.stride(), v4.stride()
        # S[b,h,q,key] = scale * q[b,q,h,:] . k[b,key,h,:]
        k_.gemm(q4, (sq[0], sq[1], 1), k4, (sk[0], sk[1], 1), P, (H * Lq * Lk, Lk, 1), Lq, Lk, d, s2=(sq[2], sk[2], Lq * Lk),
                alpha=scale, **bh)
        k_.chk(k_.lib.cgg_attn_softmax_rows(k_.h, _p(P), _p(bitmap), _p(all_masked), B, H, Lq, Lk, k_.s()), 'cgg_attn_softmax_rows')
        out = k_.new(B, Lq, H * d)
        # O[b,q,h,:] = sum_key P[b,h,q,key] v[b,key,h,:]
        k_.gemm(P, (H * Lq * Lk, Lk, 1), v4, (sv[0], 1, sv[1]), out, (Lq * H * d, H * d, 1), Lq, d, Lk, s2=(Lq * Lk, sv[2], d), **bh)
        ctx.k, ctx.scale = k_, scale
        ctx.save_for_backward(q4, k4, v4, P, out)
        return out

    @staticmethod
    def backward(ctx, dout):
        k_, scale = ctx.k, ctx.scale
        q4, k4, v4, P, out = ctx.saved_tensors
        B, Lq, H, d = q4.shape
        Lk = k4.shape[1]
        Cc = H * d
        dout = dout.contiguous()
        bh = dict(batch=B * H, batch_inner=H)
        sq, sk, sv = q4.stride(), k4.stride(), v4.stride()
        dS = k_.new(B, H, Lq, Lk)
        # dP[b,h,q,key] = dO[b,q,h,:] . v[b,key,h,:]
        k_.gemm(dout, (Lq * Cc, Cc, 1), v4, (sv[0], sv[1], 1), dS, (H * Lq * Lk, Lk, 1), Lq, Lk, d, s2=(d, sv[2], Lq * Lk), **bh)
        k_.chk(k_.lib.cgg_attn_dscore(k_.h, _p(P), _p(dS), _p(out), _p(dout), B, H, d, Lq, Lk, k_.s()), 'cgg_attn_dscore')
        dq, dk, dv = k_.new(B, Lq, H, d), k_.new(B, Lk, H, d), k_.new(B, Lk, H, d)
        # dq[b,q,h,:] = scale * sum_key dS k ;  dk[b,key,h,:] = scale * sum_q dS q ;  dv[b,key,h,:] = sum_q P dO
        k_.gemm(dS, (H * Lq * Lk, Lk, 1), k4, (sk[0], 1, sk[1]), dq, (Lq * Cc, Cc, 1), Lq, d, Lk, s2=(Lq * Lk, sk[2], d),
                alpha=scale, **bh)
        k_.gemm(dS, (H * Lq * Lk, 1, Lk), q4, (sq[0], 1, sq[1]), dk, (Lk * Cc, Cc, 1), Lk, d, Lq, s2=(Lq * Lk, sq[2], d),
                alpha=scale, a_mmajor=True, **bh)
        k_.gemm(P, (H * Lq * Lk, 1, Lk), dout, (Lq * Cc, 1, Cc), dv, (Lk * Cc, Cc, 1), Lk, d, Lq, s2=(Lq * Lk, d, d),
                a_mmajor=True, **bh)
        return None, dq, dk, dv, None, None, None


class _GradSink:
    """One gradient buffer shared by the nodes of a step that all contribute to the same input (the mask features feed the
    einsum of all 10 head calls): the first backward to run creates it and hands it to autograd, the later ones add into
    it in place (GEMM epilogue `accumulate`) and return nothing -- instead of 10 full-size gradients summed pairwise."""

    def __init__(self):
        self.buf = None


class _MaskEinsum(torch.autograd.Function):
    """mask_pred[b,q,p] = sum_c me[b,q,c] F[b,c,p]  (head.py:748).  me (B, Q, C), F (B, C, H4, W4)."""

    @staticmethod
    def forward(ctx, k, me, F, sink=None):
        B, Q, Cc = me.shape
        H4, W4 = F.shape[-2:]
        HW = H4 * W4
        out = k.new(B, Q, H4, W4)
        k.gemm(F, (Cc * HW, 1, HW), me, (Q * Cc, Cc, 1), out, (Q * HW, 1, HW), HW, Q, Cc, batch=B, a_mmajor=True,
               c_mmajor=True)
        ctx.k, ctx.sink = k, sink
        ctx.save_for_backward(me, F)
        return out

    @staticmethod
    def backward(ctx, dmask):
        k, sink = ctx.k, ctx.sink
        me, F = ctx.saved_tensors
        B, Q, Cc = me.shape
        H4, W4 = F.shape[-2:]
        HW = H4 * W4
        dmask = dmask.contiguous()
        dme = dF = None
        if ctx.needs_input_grad[1]:                       # dme[b,q,c] = sum_p dmask[b,q,p] F[b,c,p]
            dme = k.new(B, Q, Cc)
            k.gemm(dmask, (Q * HW, HW, 1), F, (Cc * HW, HW, 1), dme, (Q * Cc, Cc, 1), Q, Cc, HW, batch=B)
        if ctx.needs_input_grad[2]:                       # dF[b,c,p] = sum_q me[b,q,c] dmask[b,q,p]
            first = sink is None or sink.buf is None
            dst = k.new(B, Cc, H4, W4) if first else sink.buf
            k.gemm(dmask, (Q * HW, 1, HW), me, (Q * Cc, 1, Cc), dst, (Cc * HW, 1, HW), HW, Cc, Q, batch=B, a_mmajor=True,
                   c_mmajor=True, accumulate=not first)
            if first:
                dF = dst
                if sink is not None:
                    sink.buf = dst
        return None, dme, dF, None


# --------------------------------------------------------------------------------------------- the forward
def decoder_forward_train(head, mask_features, multi_scale_memorys, forced_attn_masks=None):
    """Autograd-connected `(cls_list, cls_emb_list, mask_list)` (10 entries each) of head.py:787-849, fp32.
    mask_features (B, C, H4, W4) and the three memories may require grad (they come from the pixel decoder).
    forced_attn_masks (tests only): 9 (bitmap, all_masked) pairs used INSTEAD of the masks derived from this forward's
    own logits, so that a gradient comparison cannot be derailed by one threshold-band bit of a tiny key set."""
    if not mask_features.is_cuda:
        raise _lib.CggError('the training path runs on CUDA only (no CPU fallback)')
    if head.pred_emb_norm and head.use_class_emb:
        raise _lib.CggError('pred_emb_norm with use_class_emb is not built on the training path')
    rt = head._runtime(mask_features.device)
    k = _K(rt, tf32=(head.train_precision == 'tf32'))
    mf = mask_features.float().contiguous()
    mems = [m.float().contiguous() for m in multi_scale_memorys]
    B, Cc, H4, W4 = mf.shape
    Q, L = head.num_queries, head.num_transformer_decoder_layers
    sizes = [tuple(m.shape[-2:]) for m in mems]
    H = head.num_heads
    d = Cc // H
    scale = 1.0 / math.sqrt(d)
    dec = head.transformer_decoder
    qe = head.query_embed.weight
    with torch.no_grad():
        pos = [rt.sine_pos(h, w) for (h, w) in sizes]                          # (K_l, C) constants
    prep = [_MemPrep.apply(k, mems[l], head.level_embed.weight[l], pos[l]) for l in range(3)]

    # fused weight gradients: when the parameters already carry a .grad at forward time (GradReducer.zero(), or zeroed by
    # the caller), the linear layers write dW / db into it on a side stream (see _WgradSide)
    side = _WgradSide(mask_features.device) if (head.fused_wgrad and torch.is_grad_enabled()) else None
    k.wgrad = side

    def dst(param, sl=None):
        # (only for parameters whose gradient bookkeeping is ours -- a GradReducer -- or on request: anything that relies on
        # autograd's accumulation hooks for these parameters, e.g. torch's DDP, would never see the gradient arrive)
        if side is None or param.grad is None or not param.requires_grad:
            return None
        if param not in _FUSED_REDUCERS and head.fused_wgrad != 'always':
            return None
        return side.target(param, param.grad if sl is None else param.grad[sl])

    def lin(x, m, res=None, alpha=1.0, relu=False, rows=None):
        return _Linear.apply(k, x, m.weight, m.bias, res, alpha, relu, dst(m.weight), dst(m.bias))

    def lin_in(x, attn, part, alpha=1.0):
        """One third (0 = q, 1 = k, 2 = v) of a fused nn.MultiheadAttention in-projection."""
        sl = slice(part * Cc, (part + 1) * Cc)
        return _Linear.apply(k, x, attn.in_proj_weight[sl], attn.in_proj_bias[sl], None, alpha, False,
                             dst(attn.in_proj_weight, sl), dst(attn.in_proj_bias, sl))

    def ln(x, m):
        return _LayerNorm.apply(k, x, m.weight, m.bias, 1e-5)

    def attention(q, kk, v, bm, am):
        """q (B * Q, C) scaled, k / v (B * K, C) -> (B, Q, C): the tcgen05 products in the tf32 mode, the flash-style FMA
        kernels (exact mode) in fp32."""
        if k.tf32:
            return _AttentionViews.apply(k, q.view(B, Q, H, d), kk.view(B, -1, H, d), v.view(B, -1, H, d), bm, am, 1.0)
        return _Attention.apply(k, q.view(B, Q, Cc), kk.view(B, -1, Cc), v.view(B, -1, Cc), bm, am, H)

    cls_list, emb_list, mask_list = [], [], []
    mf_sink = _GradSink()

    def head_call(x, lvl):
        """forward_head, head.py:711-761; returns the detached attention-mask bitmap for level lvl."""
        z = ln(x.view(B * Q, Cc), dec.post_norm)
        cls = lin(z, head.cls_embed).view(B, Q, -1)
        emb = lin(z, head.v2l_transform).view(B, Q, -1) if head.use_class_emb else cls
        me = lin(lin(lin(z, head.mask_embed[0], relu=True), head.mask_embed[2], relu=True), head.mask_embed[4])
        mask = _MaskEinsum.apply(k, me.view(B, Q, Cc), mf, mf_sink)
        cls_list.append(cls), emb_list.append(emb), mask_list.append(mask)
        if lvl is None:
            return None, None
        if forced_attn_masks is not None:
            return forced_attn_masks[len(mask_list) - 1]
        with torch.no_grad():                                                   # head.py:759: attn_mask.detach()
            return rt.attn_mask_from_logits(mask.detach(), sizes[lvl])

    x = _AddRows.apply(k, None, head.query_feat.weight, B)                       # head.py:808-809
    bm, am = head_call(x, 0)
    for i in range(L):
        lvl = i % 3
        layer = dec.layers[i]
        ca, sa = layer.attentions[0].attn, layer.attentions[1].attn
        key_in, val_in = prep[lvl]
        K = key_in.shape[1]
        x2d = x.view(B * Q, Cc)
        # ---- masked cross-attention (mmcv MultiheadAttention wrapper: identity + attn, value gets no pos)
        xq = _AddRows.apply(k, x, qe, B).view(B * Q, Cc)
        q = lin_in(xq, ca, 0, scale)
        kk = lin_in(key_in.view(B * K, Cc), ca, 1)
        vv = lin_in(val_in.view(B * K, Cc), ca, 2)
        o = attention(q, kk, vv, bm, am)
        t = lin(o.view(B * Q, Cc), ca.out_proj, res=x2d)
        x1 = ln(t, layer.norms[0])
        # ---- self-attention: q = k-input = x1 + query_embed, v-input = x1
        x1q = _AddRows.apply(k, x1.view(B, Q, Cc), qe, B).view(B * Q, Cc)
        q2 = lin_in(x1q, sa, 0, scale)
        k2 = lin_in(x1q, sa, 1)
        v2 = lin_in(x1, sa, 2)
        o2 = attention(q2, k2, v2, None, None)
        t2 = lin(o2.view(B * Q, Cc), sa.out_proj, res=x1)
        x2 = ln(t2, layer.norms[1])
        # ---- FFN
        f = lin(x2, layer.ffns[0].layers[0][0], relu=True)
        t3 = lin(f, layer.ffns[0].layers[1], res=x2)
        x = ln(t3, layer.norms[2]).view(B, Q, Cc)
        bm, am = head_call(x, (i + 1) % 3 if i + 1 < L else None)
    return cls_list, emb_list, mask_list


# ------------------------------------------------------------------------------------ gradient all-reduce
class GradReducer:
    """Bucketed NCCL all-reduce of the head's gradients, overlapped with the backward (data-parallel training,
    BASELINE.json configs[3]; reference: DDP built at open_set/apis/train.py:156-161).

    Parameters are packed, in reverse registration order (the order the backward produces them), into flat fp32 buckets
    of ~`bucket_mb`, and every `.grad` IS a view of its bucket slice: the backward accumulates straight into the
    buckets, no copy.  A `post_accumulate_grad` hook launches a bucket's all-reduce on a side stream as soon as its
    last gradient has arrived; `finish()` joins the side stream and divides by the world size.  `zero()` clears the
    buckets at the start of a step.  Everything is stream work, so the whole step -- forward, backward, the overlapped
    collectives -- can be captured in one CUDA graph (`GraphedStep`).  `exposed()` is the time between the end of the
    backward on the main stream and the end of the last all-reduce: the part of the communication that was NOT hidden
    (eager steps only; events cannot be timed inside a graph)."""

    def __init__(self, params, bucket_mb=8.0, group=None):
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.params = [p for p in params if p.requires_grad]
        dev = self.params[0].device
        self.cuda = dev.type == 'cuda'
        self.stream = torch.cuda.Stream(dev) if self.cuda else None
        self.buckets = []            # dict(flat, params[(p, off)], pending)
        cap = int(bucket_mb * (1 << 20) / 4)
        cur, n = [], 0
        for p in reversed(self.params):
            if cur and n + p.numel() > cap:
                self._close(cur, n, dev)
                cur, n = [], 0
            cur.append((p, n))
            n += p.numel()
        if cur:
            self._close(cur, n, dev)
        self.index = {}
        for bi, bk in enumerate(self.buckets):
            for p, off in bk['params']:
                self.index[p] = (bi, off)
                p.grad = bk['flat'][off:off + p.numel()].view_as(p)
        self.handles = [p.register_post_accumulate_grad_hook(self._hook) for p in self.params]
        for p in self.params:
            _FUSED_REDUCERS[p] = self          # gradients written outside autograd (_WgradSide) report here
        self.t_bwd_end = self.t_comm_end = None
        self.timing = True
        self.reset()

    def _close(self, cur, n, dev):
        self.buckets.append(dict(flat=torch.zeros(n, dtype=torch.float32, device=dev), params=list(cur), pending=0, work=None))

    def reset(self):
        for bk in self.buckets:
            bk['pending'] = len(bk['params'])
            bk['work'] = None
            bk['producers'] = set()
            bk['reported'] = set()

    def zero(self):
        """Start of a step: clear the buckets (the backward accumulates into them) and re-attach any .grad that was
        replaced (`p.grad = None`, an optimizer's set_to_none)."""
        for bk in self.buckets:
            bk['flat'].zero_()
            for p, off in bk['params']:
                view = bk['flat'][off:off + p.numel()].view_as(p)
                if p.grad is None or p.grad.data_ptr() != view.data_ptr():
                    p.grad = view

    def param_done(self, p, stream):
        """A gradient written straight into the bucket by kernels on `stream` (fused weight gradients) is complete."""
        self._hook(p, producer=stream)

    def _hook(self, p, producer=None):
        bi, off = self.index[p]
        bk = self.buckets[bi]
        # A parameter reports ONCE per step.  One whose gradient was written by the fused path (param_done) is reported a
        # second time by autograd: the engine still runs the parameter's accumulation node -- after every node that feeds
        # it, hence after the last fused product was enqueued -- and its post-accumulate hook fires although the gradient
        # it was handed is undefined.  Counting that report would launch the bucket's all-reduce before other gradients
        # of the bucket are complete (seen as wrong averages on 2 GPUs; harmless on one, where nothing is reduced).
        if id(p) in bk['reported']:
            return
        bk['reported'].add(id(p))
        if p.grad.data_ptr() != bk['flat'].data_ptr() + 4 * off:       # the caller replaced .grad: fold it back in
            bk['flat'][off:off + p.numel()].copy_(p.grad.reshape(-1))
            p.grad = bk['flat'][off:off + p.numel()].view_as(p)
        if producer is not None:
            bk.setdefault('producers', set()).add(producer)
        bk['pending'] -= 1
        if bk['pending'] == 0 and self.world > 1:
            if self.cuda:
                self.stream.wait_stream(torch.cuda.current_stream())
                for st in bk.get('producers', ()):
                    self.stream.wait_stream(st)
                with torch.cuda.stream(self.stream):
                    bk['work'] = dist.all_reduce(bk['flat'], group=self.group, async_op=True)
            else:
                bk['work'] = dist.all_reduce(bk['flat'], group=self.group, async_op=True)

    def finish(self):
        """Call after loss.backward(): joins the collectives and averages."""
        capturing = self.cuda and torch.cuda.is_current_stream_capturing()
        if self.cuda and self.timing and not capturing:
            self.t_bwd_end = torch.cuda.Event(enable_timing=True)
            self.t_bwd_end.record(torch.cuda.current_stream())
        launched = False
        for bk in self.buckets:
            if bk['work'] is not None:
                bk['work'].wait()
                launched = True
        if self.cuda:
            if launched:                       # (the side stream is part of the step only when a collective ran on it)
                torch.cuda.current_stream().wait_stream(self.stream)
            if self.timing and not capturing:
                self.t_comm_end = torch.cuda.Event(enable_timing=True)
                self.t_comm_end.record(torch.cuda.current_stream())
        if self.world > 1:
            for bk in self.buckets:
                bk['flat'].div_(self.world)
        self.reset()

    def exposed(self):
        if not self.cuda or self.t_bwd_end is None:
            return 0.0
        torch.cuda.synchronize()
        return self.t_bwd_end.elapsed_time(self.t_comm_end)

    def remove(self):
        for h in self.handles:
            h.remove()
        for p in self.params:
            if _FUSED_REDUCERS.get(p) is self:
                del _FUSED_REDUCERS[p]


class GraphedStep:
    """One training step -- forward, loss, backward and (with a GradReducer) the overlapped gradient all-reduce --
    captured once as a CUDA graph and replayed: the step is ~2000 small launches, and at 2 images per GPU the host
    cannot issue them as fast as the device retires them.

    `step_fn()` computes the loss from tensors the caller keeps alive and overwrites in place between steps (the static
    inputs) and returns it; it must not synchronise.  Gradients land in the parameters' `.grad` (the reducer's buckets
    when one is given) after every `replay()`; `self.loss` is the static loss tensor.  No autograd graph over these
    parameters that was built on another stream may still be alive at construction (drop old loss tensors first): its
    AccumulateGrad nodes are bound to that stream and cannot join the capture."""

    def __init__(self, step_fn, params, reducer=None, warmup=3):
        self.params = [p for p in params if p.requires_grad]
        self.reducer = reducer
        self.step_fn = step_fn
        dev = self.params[0].device
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):            # warm-up off the default stream: sizes every lazily grown buffer
            for _ in range(warmup):
                self._one()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        if reducer is None:
            for p in self.params:
                p.grad = None                     # the captured backward allocates .grad from the graph's pool
        self.graph = torch.cuda.CUDAGraph()
        with _lib.no_gc_during_capture(), torch.cuda.graph(self.graph):
            self.loss = self._one()

    def _one(self):
        if self.reducer is not None:
            self.reducer.zero()
        elif not torch.cuda.is_current_stream_capturing():
            for p in self.params:
                p.grad = None
        loss = self.step_fn()
        loss.backward()
        if self.reducer is not None:
            self.reducer.finish()
        return loss.detach()

    def replay(self):
        self.graph.replay()
        return self.loss
