#!/usr/bin/env python
"""Benchmark of the CGG decoder-head hot path (BASELINE.json metric: decoder-head images/s at
1024x1024).  One "step" = one pass of the path (Mask2FormerHeadOpen.forward after the pixel
decoder, open_set/models/mask2former_head.py:787-849) over one batch of synthetic pixel-decoder
outputs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--batch B_per_gpu] [--precision bf16|fp32] [--queries Q] [--dump-outputs DIR]

N>1 is launched by torch.distributed.run, one rank per GPU; images shard by batch, no data-path
collective (SURVEY.md section 8e), so "scaling" is weak.  Rank 0 prints ONE JSON line.  Besides the
contract's keys the line carries, each measured in the same run:
  roofline          dominant kernel (mask einsum) against BOTH roofs, timed in a sustained loop
  sustained         the device-resident leg repeated for >= 2 s (clocks sampled)
  strong_scaling    BASELINE configs[2]: global batch 64 split 64/N per GPU
  train             BASELINE configs[3]: OSPS head (Q=200, 118 classes) forward + backward with the grounding loss,
                    NCCL gradient all-reduce at N GPUs, exposed communication time
  grounding         the K7 grounding-loss stage alone (forward + backward)
  torch_gpu_baseline  (N=1) the same path as plain torch CUDA ops (what the reference executes), fp32 and bf16 autocast
  cpu_baseline      (N=1) the reference's CPU path on the host cores
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = 'decoder_head_images_per_sec_1024'
UNIT = 'images/s'
H = W = 1024
C = 256
FFN = 2048
D_L = 768
NCLS1 = 49
LAYERS = 9
DUMP_BYTES = 60 * 10**6         # --dump-outputs: at most this much in all, float32


def flops_per_image(Q, height=H, width=W):
    """Dense algorithmic FLOPs of the path per image (SURVEY.md section 8d)."""
    HW4 = (height // 4) * (width // 4)
    Ks = [(height // s) * (width // s) for s in (32, 16, 8)]
    f = (LAYERS + 1) * (2 * Q * C * HW4 + 2 * Q * C * (3 * C + D_L + NCLS1))
    for i in range(LAYERS):
        K = Ks[i % 3]
        f += 4 * Q * C * C + 4 * K * C * C + 4 * Q * K * C
    f += LAYERS * (8 * Q * C * C + 4 * Q * Q * C)
    f += LAYERS * (4 * Q * C * FFN)
    return float(f)


def dump_outputs(out_dir, outs):
    """Writes what one step of the path returned -- the cls / emb / mask lists of the head calls, each list stacked into
    one array -- as out_dir/{cls,emb,mask}.npy in float32, so that two builds can be compared output for output.  An
    array larger than its even share of DUMP_BYTES is replaced by a fixed sample of its flattened elements: the array is
    cut into cap blocks that together cover it to the last element (block i starts at floor(i * numel / cap)), and one
    element is taken from each block at a seeded offset -- the same positions on every run with the same shapes."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    cap = DUMP_BYTES // 4 // len(outs)
    for name, xs in zip(('cls', 'emb', 'mask'), outs):
        a = torch.stack([x for x in xs if x is not None])           # (--final-mask-only: the last mask only)
        if a.numel() > cap:
            starts = torch.arange(cap + 1) * a.numel() // cap
            offs = torch.randint(0, 2**62, (cap,), generator=torch.Generator().manual_seed(0)) % (starts[1:] - starts[:-1])
            a = a.reshape(-1)[(starts[:-1] + offs).to(a.device)]
        np.save(os.path.join(out_dir, name + '.npy'), a.float().cpu().numpy())


def einsum_flops_per_launch(Q, batch):
    return 2.0 * Q * C * (H // 4) * (W // 4) * batch


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d['hbm_gbs'], tflops=d.get('bf16_tflops_sustained', d['bf16_tflops']),
                    tflops_burst=d['bf16_tflops'], source='MEASURED_PEAKS.json')
    return dict(hbm_gbs=6650.0, tflops=1400.0, tflops_burst=1590.0, source='fallback (B200_PROFILING.md)')


class ClockSampler:
    """SM clock, power and throttle reasons sampled DURING the timed region: an NVML polling thread (a query is ~0.1 ms,
    so even the 50 ms K-step region of 8 concurrent ranks gets samples; `nvidia-smi -lms` cannot promise one)."""
    REASONS = ((0x8, 'hw_slowdown'), (0x40, 'hw_thermal_slowdown'), (0x20, 'sw_thermal_slowdown'), (0x4, 'sw_power_cap'))

    def __init__(self, index):
        self.index = index
        self.thread = None
        self.samples = []
        self.stop_flag = False
        self.err = None

    def _run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            get_reasons = getattr(pynvml, 'nvmlDeviceGetCurrentClocksEventReasons', None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            while True:
                self.samples.append((pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM), mx,
                                     pynvml.nvmlDeviceGetPowerUsage(h) / 1e3, int(get_reasons(h))))
                if self.stop_flag:          # (checked after sampling: a region shorter than one period still gets one)
                    break
                time.sleep(0.002)
        except Exception as e:      # noqa: BLE001
            self.err = repr(e)[:120]

    def start(self):
        import threading
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def stop(self):
        self.stop_flag = True
        if self.thread is not None:
            self.thread.join(timeout=5)
        if not self.samples:
            return dict(sm_mhz=None, sm_max_mhz=None, power_w_max=None, samples=0, reasons=['nvml unavailable: %s' % self.err])
        sm = sorted(x[0] for x in self.samples)
        bits = 0
        for x in self.samples:
            bits |= x[3]
        return dict(sm_mhz=float(sm[len(sm) // 2]), sm_max_mhz=float(self.samples[0][1]),
                    power_w_max=max(x[2] for x in self.samples), samples=len(sm),
                    reasons=sorted(n for m, n in self.REASONS if bits & m))


def trace(msg):
    if os.environ.get('CGG_BENCH_TRACE'):
        sys.stderr.write('[bench %s rank %s] %s\n' % (time.strftime('%H:%M:%S'), os.environ.get('RANK', '0'), msg))
        sys.stderr.flush()


def reduce_max(value, world, device):
    """MAX over ranks of a per-rank scalar (the timing rule: slowest rank defines the step)."""
    import torch.distributed as dist
    t = torch.tensor([value], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def whole_job_value(world, batch_per_gpu, steps, ms):
    """images/s of the whole job: every rank processed batch_per_gpu images per step (batch-sharded, no
    data-path collective -- SURVEY.md section 8e)."""
    return world * batch_per_gpu * steps / (ms * 1e-3)


def dist_env():
    return int(os.environ.get('RANK', 0)), int(os.environ.get('LOCAL_RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))


def cpu_model():
    try:
        for line in open('/proc/cpuinfo'):
            if line.startswith('model name'):
                return line.split(':', 1)[1].strip()
    except Exception:
        pass
    return 'unknown'


def pin_to_gpu_numa_node(local_rank):
    """e2e staging: pinned host buffers are first-touch allocated, so each rank first moves itself onto the CPUs next
    to its GPU (round-1 SCALE: all ranks on NUMA 0 capped the 8-GPU e2e leg at 120 GB/s aggregate)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        n = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n)
        cpus = [64 * i + b for i, word in enumerate(mask) for b in range(64) if (word >> b) & 1]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


# ------------------------------------------------------------------------------ CPU legs
def _reference_head(Q):
    """The UNMODIFIED reference head (oracle/_ref or /root/reference through the dependency shim) with the seeded
    weights, or None when no copy of the reference is available (then the oracle port is timed)."""
    try:
        from oracle import ref_shim
        if not ref_shim.reference_available():
            return None
        R = ref_shim.REF_ROOT
        head = ref_shim.build_reference_head(num_queries=Q, known_file=R + '/datasets/unknown/known_65.txt',
                                             unknown_file=R + '/datasets/unknown/unknown_17.txt')
        return head, ref_shim
    except Exception as e:      # noqa: BLE001  (a broken copy must not take the bench line down)
        sys.stderr.write('reference head unavailable (%s); timing the oracle port\n' % e)
        return None


def cpu_path(Q):
    """Returns (kind, step(mf, mems)) for the reference's CPU path."""
    from cgg_b200 import synth
    sd = synth.make_params(seed=0, num_queries=Q)
    ref = _reference_head(Q)
    if ref is not None:
        head, shim = ref
        head.load_state_dict(sd, strict=True)
        return 'reference', lambda mf, mems: shim.run_reference_head(head, mf, mems)
    from oracle import cgg_oracle as O

    def step(mf, mems):
        with torch.no_grad():
            return O.decoder_forward(sd, mf, mems)
    return 'port', step


def _time_cpu(step, mf, mems, repeats):
    step(mf, mems)
    ts = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        step(mf, mems)
        ts.append(time.perf_counter() - t0)
    ts.sort()
    return ts[len(ts) // 2]


def cpu_baseline(Q, threads):
    """The reference's fp32 PyTorch path on the host cores, bounded samples of the same workload: one 1024x1024 image
    per pass on all cores (median of 3) and on one thread (1 pass), and one batch-16 pass on all cores."""
    from cgg_b200 import synth
    kind, step = cpu_path(Q)
    torch.set_num_threads(threads)
    mf, mems = synth.make_inputs(0, 1, H, W)
    t_b1 = _time_cpu(step, mf, mems, 3)
    mf16, mems16 = synth.make_inputs(0, 16, H, W)
    t0 = time.perf_counter()
    step(mf16, mems16)
    t_b16 = time.perf_counter() - t0
    del mf16, mems16
    torch.set_num_threads(1)
    t0 = time.perf_counter()
    step(mf, mems)
    t_1t = time.perf_counter() - t0
    torch.set_num_threads(threads)
    return dict(value=1.0 / t_b1, unit=UNIT, cores=threads, kind=kind, cpu_model=cpu_model(),
                b16_value=16.0 / t_b16, single_thread_value=1.0 / t_1t,
                sample='Q=%d fp32 1024x1024: value = 1 image per pass, median of 3 after 1 warm-up, %d threads; b16_value = one '
                       'batch-16 pass; single_thread_value = 1 image, 1 thread, 1 pass' % (Q, threads))


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path (verbatim head from oracle/_ref through
    the mmcv/mmdet shim; the oracle port only if that copy is missing) with all host threads, each step a bounded
    sample of the workload: ONE 1024x1024 image."""
    rank, _, world = dist_env()
    if rank != 0:
        return
    from cgg_b200 import synth
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    Q = args.queries
    sample_b = 1
    kind, step = cpu_path(Q)
    mf, mems = synth.make_inputs(0, sample_b, H, W)
    for _ in range(min(args.warmup, 1)):
        step(mf, mems)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step(mf, mems)
    dt = time.perf_counter() - t0
    val = sample_b * args.steps / dt
    # one batch-16 pass as well (the GPU arm's batch), reported beside the per-image number
    mf16, mems16 = synth.make_inputs(0, 16, H, W)
    t0 = time.perf_counter()
    step(mf16, mems16)
    b16 = 16.0 / (time.perf_counter() - t0)
    line = dict(metric=METRIC, value=val, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=min(args.warmup, 1),
                ms_per_step=1e3 * dt / args.steps, higher_is_better=True, scaling='weak', vs_baseline=None,
                dtype='f32', data='synthetic', impl='reference',
                config=dict(workload='configs[1]: COCO-OVIS instance decoder head, Q=%d, 9 layers, 256-d, 1024x1024' % Q,
                            batch_per_step=sample_b, note='CPU path, bounded sample of 1 image per step'),
                cpu_baseline=dict(value=val, unit=UNIT, cores=threads, kind=kind, cpu_model=cpu_model(), b16_value=b16,
                                  sample='%d image(s) 1024x1024 per step, fp32, %s; b16_value = one batch-16 pass' %
                                         (sample_b, 'the unmodified reference head (oracle/_ref) under the mmcv/mmdet shim'
                                          if kind == 'reference' else 'oracle port of the reference path')),
                e2e=dict(value=val, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


# ------------------------------------------------------------------------ side legs of our arm
def torch_gpu_baseline(Q, B, dev):
    """The same path as plain torch CUDA ops -- the oracle moved to the GPU, i.e. cuBLAS / ATen kernels, which is
    what the reference executes on a GPU -- in fp32 and under bf16 autocast (BASELINE.md section 3; the >= 10x target is
    against the faster of the two)."""
    from oracle import cgg_oracle as O
    from cgg_b200 import synth
    sd = {k: v.to(dev) for k, v in synth.make_params(seed=0, num_queries=Q).items()}
    mf, mems = synth.make_inputs(0, B, H, W)
    mf, mems = mf.to(dev), [m.to(dev) for m in mems]
    out = {}
    for name, ctx in (('fp32', torch.autocast('cuda', enabled=False)), ('bf16_autocast', torch.autocast('cuda', torch.bfloat16))):
        with torch.no_grad(), ctx:
            for _ in range(2):
                O.decoder_forward(sd, mf, mems)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n = 5
            e0.record()
            for _ in range(n):
                O.decoder_forward(sd, mf, mems)
            e1.record()
            torch.cuda.synchronize()
        out[name] = B * n / (e0.elapsed_time(e1) * 1e-3)
    out.update(unit=UNIT, batch=B, note='oracle (plain torch ops) on the same GPU, 2 warm-up + 5 timed forwards, CUDA events')
    return out


def grounding_leg(dev, Bg=16, Q=100, T=35, D=768):
    """K7 alone: the caption-grounding loss of one head call for Bg images x Bg captions (reference batch 2 x 8 GPUs),
    forward + backward; algorithmic FLOPs = the similarity contraction 2 (Bg T)(Bg Q) D, x2 for the backward."""
    from cgg_b200.grounding import grounding_loss
    g = torch.Generator().manual_seed(3)
    pred = torch.randn((Bg, Q, D), generator=g).to(dev).requires_grad_(True)
    cap = (torch.randn((Bg, T, D), generator=g) * 0.85).to(dev)
    m = torch.zeros((Bg, T), dtype=torch.long)
    for b in range(Bg):
        m[b, :(3 * b) % 11] = 1
    m = m.to(dev)
    for _ in range(3):
        grounding_loss(pred, cap, m, 10.0, 2.0).backward()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 20
    e0.record()
    for _ in range(n):
        pred.grad = None
        grounding_loss(pred, cap, m, 10.0, 2.0).backward()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    fl = 2.0 * (Bg * T) * (Bg * Q) * D * 3      # forward S, backward recompute of S, dpred contraction
    return dict(ms_fwd_bwd=ms, Bg=Bg, Q=Q, tokens=T, tflops=fl / (ms * 1e-3) / 1e12,
                note='cgg_grounding_loss + cgg_grounding_loss_backward, one head call, fp32')


def pixel_decoder_leg(dev, B, head=None, precision='tf32', steps=5):
    """Row f3 alone, then chained: mmdet's MSDeformAttnPixelDecoder (the step before the path, head.py:787) at the configs[1]
    shapes -- B images of 1024^2, R50 channel widths (256/512/1024/2048 at strides 4..32), 6 encoder layers -- through
    cgg_b200.pixel_decoder (every contraction on tcgen05 kind::tf32), and the same step as plain torch CUDA ops (the oracle on
    the GPU: cuDNN convs, ATen GroupNorm / grid_sample -- mmcv's pure-torch deformable attention).  Algorithmic FLOPs: the
    contractions only."""
    from cgg_b200 import synth
    from cgg_b200.pixel_decoder import build_pixel_decoder_from_state_dict
    from oracle import pixel_decoder_oracle as PO
    chs = (256, 512, 1024, 2048)
    sd = synth.make_pixel_decoder_params(0, in_channels=chs)
    feats = [f.to(dev) for f in synth.make_backbone_feats(0, B, H, W, chs)]
    m = build_pixel_decoder_from_state_dict(sd, chs, dev, precision=precision).eval()

    def timed(fn, n, w=2):
        for _ in range(w):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    S = sum((H // s) * (W // s) for s in (32, 16, 8))
    P4 = (H // 4) * (W // 4)
    fl = 2.0 * 256 * sum(c * (H // s) * (W // s) for c, s in zip(chs[1:], (8, 16, 32)))          # input convs
    fl += 6 * 2.0 * S * (256 * (256 + 192 + 96 + 256) + 2 * 256 * 1024)                         # encoder linears
    fl += 2.0 * P4 * 256 * (chs[0] + 9 * 256 + 256)                                             # lateral, 3x3 output conv, mask conv
    out = dict(batch=B, precision=precision, tokens_per_image=S, gflop_per_image=fl / 1e9)
    with torch.no_grad():
        ms = timed(lambda: m(feats), steps)
        out.update(ms=ms, images_per_s=B / ms * 1e3, tflops=fl * B / (ms * 1e-3) / 1e12)
        if head is not None:                     # pixel decoder -> decoder head in one call (Mask2FormerHeadOpenB200.forward)
            m.out_dtype = torch.bfloat16 if head.precision == 'bf16' else torch.float32
            head.pixel_decoder = m
            metas = [dict()] * B
            ms2 = timed(lambda: head(feats, metas), steps)
            head.pixel_decoder = None
            out['with_decoder_head'] = dict(ms=ms2, images_per_s=B / ms2 * 1e3,
                                            note='Mask2FormerHeadOpenB200.forward(feats, img_metas): pixel decoder + the '
                                                 '10-head-call decoder path, eager launches, one batch in flight')
        sd_d = {k: v.to(dev) for k, v in sd.items()}
        base = {}
        for name, tf32 in (('fp32', False), ('tf32', True)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            base[name + '_ms'] = timed(lambda: PO.pixel_decoder_forward(sd_d, feats), 3, 1)
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = True
        out['torch_gpu_baseline'] = base
        out['speedup_vs_faster'] = min(base.values()) / ms
    # ---- training form: forward + backward at the configs[3] batch (2 images per GPU), gradients to every parameter and to
    # the backbone maps, against the same step as plain torch CUDA ops + autograd
    try:
        Bt = 2
        ft = [f[:Bt].clone().requires_grad_(True) for f in feats]
        m.out_dtype = torch.float32
        m.train()

        def ours():
            for p_ in m.parameters():
                p_.grad = None
            mf, mems = m(ft)
            (mf.square().mean() + sum(t.square().mean() for t in mems)).backward()

        sd_g = {k: v.to(dev).requires_grad_(True) for k, v in sd.items()}

        def plain():
            for v in sd_g.values():
                v.grad = None
            mf, mems = PO.pixel_decoder_forward(sd_g, ft)
            (mf.square().mean() + sum(t.square().mean() for t in mems)).backward()

        torch.backends.cuda.matmul.allow_tf32 = True
        out['train_step'] = dict(batch=Bt, ms_fwd_bwd=timed(ours, 3, 2), torch_tf32_ms_fwd_bwd=timed(plain, 3, 1))
        torch.backends.cuda.matmul.allow_tf32 = False
        m.eval()
    except Exception as e:      # noqa: BLE001
        out['train_step'] = dict(error=repr(e)[:300])
    out['note'] = ('cgg_b200.pixel_decoder.MSDeformAttnPixelDecoderB200 forward, token-major fp32 activations, contractions on '
                   'tcgen05 kind::tf32; inputs resident in HBM (%.0f MB per step)' % (sum(f.numel() for f in feats) * 4 / 1e6))
    return out


def matching_leg(dev, B=2, Q=200, ncls1=118, G=20, h=256, w=256, P=12544):
    """Row f2 alone: the matching-based terms of loss_single for ONE head call at the configs[3] shapes (B images, Q
    queries, G ground-truth masks per image, 12 544 points): point sampling, cost matrix, Hungarian solve (host),
    class-weighted CEs, importance-sampled dice + BCE, forward + backward; the same function as plain torch CUDA ops
    (the oracle moved to the GPU, its Hungarian solve on the host too) beside it."""
    import time
    from cgg_b200 import synth, matching
    from cgg_b200.head import build_head_from_state_dict
    from oracle import matching_oracle as MO
    head = build_head_from_state_dict(synth.make_params(seed=0, num_queries=Q, num_classes_p1=ncls1), Q, ncls1, 'fp32', dev)
    ml = matching.MatchingLosses(head, train_cfg=dict(num_points=P))
    g = torch.Generator().manual_seed(4)
    mask = (torch.randn((B, Q, h, w), generator=g) * 2).to(dev).requires_grad_(True)
    cls = torch.randn((B, Q, ncls1), generator=g).to(dev).requires_grad_(True)
    emb = (torch.randn((B, Q, ncls1), generator=g) * 2).to(dev).requires_grad_(True)
    gt_labels = [torch.randint(0, ncls1 - 1, (G,), generator=g).to(dev) for _ in range(B)]
    gt_masks = []
    for _ in range(B):
        m = torch.zeros((G, h, w))
        for k in range(G):
            y0, x0 = int(torch.randint(0, h // 2, (1,), generator=g)), int(torch.randint(0, w // 2, (1,), generator=g))
            m[k, y0:y0 + h // 4, x0:x0 + w // 4] = 1.0
        gt_masks.append(m.to(dev))

    def ours():
        out, _, _ = ml.loss_single(cls, emb, mask, gt_labels, gt_masks)
        (out['loss_cls_emb'] + out['loss_mask'] + out['loss_dice']).backward()

    def plain():
        out = MO.loss_single_matching(cls, emb, mask, gt_labels, gt_masks, ncls1 - 1, dict(num_points=P))
        (out['loss_cls_emb'] + out['loss_mask'] + out['loss_dice']).backward()

    res = {}
    for name, fn in (('ms_fwd_bwd', ours), ('torch_gpu_ms_fwd_bwd', plain)):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n = 5
        for _ in range(n):
            mask.grad = cls.grad = emb.grad = None
            fn()
        torch.cuda.synchronize()
        res[name] = (time.perf_counter() - t0) / n * 1e3
    res.update(images=B, queries=Q, gts_per_image=G, points=P,
               note='wall clock per call (the Hungarian solve and the positives gather synchronise with the host, as in '
                    'the reference); one head call, fp32')
    return res


def train_leg(args, rank, world, dev):
    """BASELINE configs[3]: OSPS head (200 queries, 118 class rows), forward + backward of the decoder head with the
    caption-grounding loss on every head call (weight 2.0) + class-embedding CE + a point-sampled mask BCE, per-GPU batch 2
    (coco_panoptic_p20.py:236), bucketed NCCL all-reduce of the 14.7 M head gradients overlapped with the backward.
    Contractions on tcgen05 (kind::tf32), the whole step replayed as one CUDA graph; the same step issued eagerly and
    the same step as plain torch CUDA ops (the oracle on the GPU, TF32 matmuls: what the reference executes) beside it."""
    import torch.distributed as dist
    from cgg_b200 import synth
    from cgg_b200.head import build_head_from_state_dict
    from cgg_b200.grounding import grounding_loss, gather_captions_and_preds, similarity
    from cgg_b200.train import GradReducer, GraphedStep
    Q, B, ncls1 = 200, args.train_batch, 118
    sd = synth.make_params(seed=0, num_queries=Q, num_classes_p1=ncls1)
    head = build_head_from_state_dict(sd, Q, ncls1, 'fp32', dev, train_precision=args.train_precision).train()
    mf, mems = synth.make_inputs(100 + rank, B, H, W)
    mf, mems = mf.to(dev), [m.to(dev) for m in mems]
    ids, cap_mask, table, lw, lb = synth.make_captions(rank, B)
    cap = head.extract_word_embeddings(table.to(dev), lw.to(dev), lb.to(dev), ids.to(dev))
    cap_mask = cap_mask.to(dev)
    g = torch.Generator().manual_seed(rank)
    labels = torch.randint(0, ncls1, (B, Q), generator=g).to(dev)
    # mask surrogate: BCE on 12 544 points sampled from every query's mask logits (the reference's mask losses are
    # point-sampled too, head.py:600-627; its Hungarian matching needs the host and is timed separately below)
    from cgg_b200.matching import point_sample
    coords = torch.rand((1, 12544, 2), generator=g).to(dev)
    targets = (torch.rand((B * Q, 12544), generator=g) > 0.5).to(dev).float()
    reducer = GradReducer(head.parameters())
    ce, bce = torch.nn.functional.cross_entropy, torch.nn.functional.binary_cross_entropy_with_logits

    def loss_fn():
        cls, emb, mask = head.decoder_forward_auto(mf, mems)
        loss = 0.0
        embs_all, mask_all, preds_all = gather_captions_and_preds(cap, cap_mask, torch.stack(emb, 0))
        for j in range(len(cls)):
            loss = loss + grounding_loss(preds_all[j], embs_all, mask_all, 10.0, 2.0)
            loss = loss + ce(similarity(emb[j].reshape(B * Q, -1), head.class_embs, 0.1), labels.reshape(-1))
            loss = loss + bce(point_sample(mask[j].view(B * Q, H // 4, W // 4), coords), targets)
        return loss

    def eager_step():
        reducer.zero()
        loss_fn().backward()
        reducer.finish()

    def timed(fn, n, after=None):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        extra = 0.0
        e0.record()
        for _ in range(n):
            fn()
            if after:
                extra += after()
        e1.record()
        torch.cuda.synchronize()
        return reduce_max(e0.elapsed_time(e1) / n, world, dev), extra / n

    # the reference's full loss dict (grounding + Hungarian-matched class / mask / dice terms, row f2): the assignment
    # synchronises with the host (scipy, as in the reference), so this form of the step cannot be one CUDA graph
    from cgg_b200.matching import MatchingLosses
    ml = MatchingLosses(head, train_cfg=dict(num_points=12544))
    G = 20
    gt_labels = [torch.randint(0, ncls1 - 1, (G,), generator=g).to(dev) for _ in range(B)]
    gt_masks = []
    for _ in range(B):
        m = torch.zeros((G, H // 4, W // 4))
        for k in range(G):
            y0, x0 = int(torch.randint(0, H // 8, (1,), generator=g)), int(torch.randint(0, W // 8, (1,), generator=g))
            m[k, y0:y0 + H // 16, x0:x0 + W // 16] = 1.0
        gt_masks.append(m.to(dev))

    def full_loss_step():
        reducer.zero()
        cls, emb, mask = head.decoder_forward_auto(mf, mems)
        embs_all, mask_all, preds_all = gather_captions_and_preds(cap, cap_mask, torch.stack(emb, 0))
        loss = sum(grounding_loss(preds_all[j], embs_all, mask_all, 10.0, 2.0) for j in range(len(cls)))
        loss = loss + sum(ml(cls, emb, mask, gt_labels, gt_masks).values())
        loss.backward()
        reducer.finish()

    n = args.train_steps
    trace('train: setup done')
    for _ in range(2):
        full_loss_step()
    trace('train: full-loss warm-up done')
    full_ms, _ = timed(full_loss_step, n)
    trace('train: full-loss timed')
    for _ in range(2):
        eager_step()
    trace('train: eager warm-up done')
    eager_ms, exposed = timed(eager_step, n, after=reducer.exposed)
    trace('train: eager timed')
    exposed = reduce_max(exposed, world, dev)
    out = dict(batch_per_gpu=B, queries=Q, classes_p1=ncls1, precision=args.train_precision,
               grad_bytes=4 * sum(p.numel() for p in head.parameters()),
               eager=dict(ms_per_step=eager_ms, allreduce_exposed_ms=exposed,
                          note='issued launch by launch; exposed = end of backward -> end of the last bucket all-reduce'),
               full_loss_eager=dict(ms_per_step=full_ms, gts_per_image=G, points=12544,
                                    note='grounding x10 + Hungarian-matched loss_cls / loss_cls_emb / loss_mask / loss_dice '
                                         'x10 (cgg_b200.matching: the reference\'s full loss dict less caption generation), '
                                         'issued eagerly: the assignment synchronises with the host as in the reference'))
    ms = eager_ms
    if not args.no_train_graph:
        reducer.timing = False
        gs = GraphedStep(loss_fn, head.parameters(), reducer=reducer)
        trace('train: graph captured')
        for _ in range(2):
            gs.replay()
        trace('train: graph replayed')
        ms, _ = timed(gs.replay, max(n, 10))
        out['cuda_graph'] = True
    out.update(ms_per_step=ms, images_per_s=world * B / (ms * 1e-3),
               note='forward + backward through cgg_b200.train (every node a C-ABI kernel; contractions on tcgen05 '
                    'kind::tf32), losses: grounding x10 + class-embedding CE x10 + point-sampled mask BCE x10; optimizer step '
                    'excluded; bucketed NCCL all-reduce overlapped with the backward%s'
                    % (', the whole step one CUDA graph' if out.get('cuda_graph') else ''))
    reducer.remove()
    if rank == 0 and not args.no_torch_baseline:
        # the same step as plain torch CUDA ops: the oracle on this GPU (single process, no all-reduce)
        from oracle import cgg_oracle as O
        from oracle import matching_oracle as MO
        sd_t = {k: v.to(dev).requires_grad_(k != 'class_embs') for k, v in sd.items()}

        def torch_step():
            for v in sd_t.values():
                v.grad = None
            ref = O.decoder_forward(sd_t, mf, mems)
            loss = 0.0
            for j in range(10):
                loss = loss + O.grounding_loss(ref['emb'][j], cap, cap_mask, 10.0, 2.0)
                loss = loss + ce(O.cls_emb_logits(ref['emb'][j].reshape(B * Q, -1), sd_t['class_embs'], 10.0), labels.reshape(-1))
                loss = loss + bce(MO.point_sample(ref['mask'][j].flatten(0, 1).unsqueeze(1), coords.expand(B * Q, -1, -1)).squeeze(1),
                                  targets)
            loss.backward()

        res = {}
        old = torch.backends.cuda.matmul.allow_tf32
        try:
            for name, flag in (('fp32', False), ('tf32', True)):
                torch.backends.cuda.matmul.allow_tf32 = flag
                for _ in range(2):
                    torch_step()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(3):
                    torch_step()
                e1.record()
                torch.cuda.synchronize()
                res[name + '_ms_per_step'] = e0.elapsed_time(e1) / 3
        finally:
            torch.backends.cuda.matmul.allow_tf32 = old
        res['note'] = 'oracle (plain torch ops + autograd) on the same GPU, same losses, one process'
        res['speedup_vs_faster'] = min(res['fp32_ms_per_step'], res['tf32_ms_per_step']) / ms
        out['torch_gpu_baseline'] = res
    if world > 1:
        dist.barrier()
    return out


# ------------------------------------------------------------------------------- our arm
def run_b200_arm(args):
    import torch.distributed as dist
    from cgg_b200 import synth, lib as clib
    from cgg_b200.head import build_head_from_state_dict

    rank, local_rank, world = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device -- the B200 path has no CPU fallback')
    numa_cpus = pin_to_gpu_numa_node(local_rank) if world > 1 else 0
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    Q, B = args.queries, args.batch
    dt_in = torch.bfloat16 if args.precision == 'bf16' else torch.float32
    sd = synth.make_params(seed=0, num_queries=Q)
    head = build_head_from_state_dict(sd, Q, NCLS1, args.precision, dev, cuda_graph=not args.no_graph,
                                      final_mask_only=args.final_mask_only)
    # synthetic pixel-decoder outputs, per-rank seed; kept in PINNED host memory for the e2e leg
    mf_h, mems_h = synth.make_inputs(rank, B, H, W, dtype=dt_in)
    mf_h = mf_h.pin_memory()
    mems_h = [m.pin_memory() for m in mems_h]
    mf_d = mf_h.to(dev, non_blocking=True)
    mems_d = [m.to(dev, non_blocking=True) for m in mems_h]
    lib = clib.load()

    # `value` keeps args.in_flight batches in flight: one head (own workspace, own CUDA graph) and one stream per
    # slot, steps issued round-robin.  The layer chain of a step is latency-bound (DESIGN.md section 6), so the
    # chain of one batch fills the SMs the other leaves idle; every step is still a full forward of B images.
    n_fly = max(1, args.in_flight)
    heads = [head] + [build_head_from_state_dict(sd, Q, NCLS1, args.precision, dev, cuda_graph=not args.no_graph,
                                                 final_mask_only=args.final_mask_only)
                      for _ in range(n_fly - 1)]
    fly_in = [(mf_d, mems_d)] + [(mf_d.clone(), [m.clone() for m in mems_d]) for _ in range(n_fly - 1)]
    fly_streams = [torch.cuda.Stream() for _ in range(n_fly)]
    step_no = [0]
    last_out = [None]           # what the last timed step returned (--dump-outputs)

    def step_resident():
        i = step_no[0] % n_fly
        step_no[0] += 1
        with torch.cuda.stream(fly_streams[i]):
            return heads[i].decoder_forward(*fly_in[i])

    def fork():
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        for st in fly_streams:
            st.wait_event(ev)

    def join():
        for st in fly_streams:
            torch.cuda.current_stream().wait_stream(st)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        fork()
        for _ in range(n):
            last_out[0] = step_resident()
        join()
        e1.record()
        barrier()
        return e0.elapsed_time(e1)

    fork()
    for _ in range(max(args.warmup, 3) * n_fly):
        out = step_resident()
    join()
    barrier()
    # single-batch latency of one step (one stream, nothing else in flight), reported next to the throughput
    l0_, l1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0_.record()
    for _ in range(5):
        head.decoder_forward(mf_d, mems_d)
    l1_.record()
    torch.cuda.synchronize()
    latency_ms = l0_.elapsed_time(l1_) / 5
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = lib.cgg_launch_count()
    ms = timed(args.steps)
    launches = lib.cgg_launch_count() - launches0
    if launches == 0:
        # CUDA-graph replay: the host-side counter does not tick; count one eager pass of the same
        # path (identical kernel sequence to the captured one) and scale by the timed steps
        l0 = lib.cgg_launch_count()
        head._runtime(dev)._forward_eager(mf_d, mems_d)
        torch.cuda.synchronize()
        launches = (lib.cgg_launch_count() - l0) * args.steps
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_out[0])
    ms = reduce_max(ms, world, dev)
    value = whole_job_value(world, B, args.steps, ms)

    # ---- sustained leg: the same loop for >= 2 s (the K-step region above lasts tens of ms at boost clocks)
    n_sus = max(args.steps, int(args.sustain_s * 1e3 / (ms / args.steps)) + 1)
    sampler2 = ClockSampler(local_rank)
    if rank == 0:
        sampler2.start()
    ms_sus = reduce_max(timed(n_sus), world, dev)
    sus_clocks = sampler2.stop() if rank == 0 else None
    trace('sustained leg done')
    sustained = dict(value=whole_job_value(world, B, n_sus, ms_sus), unit=UNIT, steps=n_sus, seconds=ms_sus * 1e-3,
                     ms_per_step=ms_sus / n_sus, clocks=sus_clocks)

    # ---- e2e: public API with HOST buffers; H2D of the step's inputs and D2H of the step's
    # result (last layer's cls / cls_emb / mask logits, what simple_test consumes, head.py:943-945)
    res_h = None
    h2d = mf_h.numel() * mf_h.element_size() + sum(m.numel() * m.element_size() for m in mems_h)

    # Three streams, double-buffered device inputs: the H2D copy of step i+1 and the D2H read of
    # step i-1 overlap the kernels of step i (PCIe is full duplex); every step still pays its own
    # H2D + D2H, and the loop ends with a full synchronise.
    main = torch.cuda.current_stream()
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    in_bufs = [(torch.empty_like(mf_d), [torch.empty_like(m) for m in mems_d]) for _ in range(2)]
    in_ready = [torch.cuda.Event() for _ in range(2)]
    in_free = [torch.cuda.Event() for _ in range(2)]
    out_free = torch.cuda.Event()

    def upload(slot):
        with torch.cuda.stream(s_in):
            s_in.wait_event(in_free[slot])
            in_bufs[slot][0].copy_(mf_h, non_blocking=True)
            for d, hsrc in zip(in_bufs[slot][1], mems_h):
                d.copy_(hsrc, non_blocking=True)
            in_ready[slot].record(s_in)

    def run_e2e(n):
        nonlocal res_h
        for e in in_free:
            e.record(main)
        out_free.record(main)
        upload(0)
        for i in range(n):
            slot = i & 1
            if i + 1 < n:
                upload(slot ^ 1)
            main.wait_event(in_ready[slot])
            cls, emb, mask = head.decoder_forward(in_bufs[slot][0], in_bufs[slot][1])
            in_free[slot].record(main)
            done = torch.cuda.Event()
            done.record(main)
            if res_h is None:
                res_h = [torch.empty(x.shape, dtype=x.dtype).pin_memory() for x in (cls[-1], emb[-1], mask[-1])]
            with torch.cuda.stream(s_out):
                s_out.wait_event(done)
                for dst, src in zip(res_h, (cls[-1], emb[-1], mask[-1])):
                    src.record_stream(s_out)
                    dst.copy_(src, non_blocking=True)
                out_free.record(s_out)
        torch.cuda.synchronize()

    run_e2e(2)
    barrier()
    e2e_steps = max(4, args.steps)
    t0 = time.perf_counter()
    run_e2e(e2e_steps)
    barrier()
    trace('e2e leg done')
    e2e_val = whole_job_value(world, B, e2e_steps, 1e3 * reduce_max(time.perf_counter() - t0, world, dev))
    d2h = sum(x.numel() * x.element_size() for x in res_h)
    del in_bufs

    # ---- strong scaling, BASELINE configs[2]: global batch 64 split evenly, 64/N images per GPU per step
    strong = None
    if args.precision == 'bf16' and not args.no_strong and 64 % world == 0:
        bs = 64 // world
        chunk = min(bs, 16)                      # N=1 runs the 64 images as 4 x 16 (SURVEY.md section 8d config 3)
        hs = head if chunk == B else build_head_from_state_dict(sd, Q, NCLS1, args.precision, dev, cuda_graph=not args.no_graph)
        mfs, memss = synth.make_inputs(1000 + rank, chunk, H, W, dtype=dt_in)
        mfs, memss = mfs.to(dev), [m.to(dev) for m in memss]
        for _ in range(3):
            hs.decoder_forward(mfs, memss)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_it = 5
        e0.record()
        for _ in range(n_it * (bs // chunk)):
            hs.decoder_forward(mfs, memss)
        e1.record()
        barrier()
        ms_s = reduce_max(e0.elapsed_time(e1) / n_it, world, dev)
        strong = dict(global_batch=64, batch_per_gpu=bs, ms_per_global_batch=ms_s, value=64.0 / (ms_s * 1e-3), unit=UNIT,
                      scaling='strong', note='configs[2]: 64 images per step over N GPUs, one batch in flight per GPU')
        del hs, mfs, memss

    # ---- roofline of the dominant kernel (the mask einsum, 55% of the path's FLOPs): CUDA events
    # on the launching stream around that stage alone, same inputs, back-to-back for >= 1 s so the clocks are the
    # SUSTAINED ones the sustained peak was measured at
    rt = head._runtime(dev)
    peaks = measured_peaks()
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if args.precision == 'bf16':
        # K2 alone: ONE launch of the tcgen05 GEMM computes the mask logits of all 10 head calls
        # (the mask embeddings of the last forward are still in the workspace); 2.1 GB of output
        # per launch, far larger than L2.
        mask_out = torch.empty((LAYERS + 1, B, Q, H // 4, W // 4), dtype=torch.bfloat16, device=dev)
        for _ in range(3):
            rt.mask_einsum(mf_d, mask_out)
        torch.cuda.synchronize()
        # (a) 10 launches back to back (~6 ms, boost clocks): the regime MEASURED_PEAKS.json's HBM copy peak and burst
        #     tensor peak were taken in ("best of 10")
        k0.record()
        for _ in range(10):
            rt.mask_einsum(mf_d, mask_out)
        k1.record()
        torch.cuda.synchronize()
        kern_ms_burst = k0.elapsed_time(k1) / 10
        # (b) back to back for >= 1 s (power-capped clocks): the regime of the sustained tensor peak
        reps = max(10, int(1000.0 / max(kern_ms_burst, 1e-3)))
        k0.record()
        for _ in range(reps):
            rt.mask_einsum(mf_d, mask_out)
        k1.record()
        torch.cuda.synchronize()
        kern_ms = k0.elapsed_time(k1) / reps
        flops = einsum_flops_per_launch(Q, B) * (LAYERS + 1)
        alg_bytes = B * C * (H // 4) * (W // 4) * 2 + (LAYERS + 1) * B * Q * (H // 4) * (W // 4) * 2
        kname = 'tc_einsum_t_kernel (cta_group::2, queries on TMEM lanes): mask einsum of all 10 head calls, one launch (cgg_mask_einsum)'
        del mask_out
    else:
        x0 = torch.randn((B, Q, C), device=dev)
        reps = 10
        for _ in range(3):
            rt.head_call(x0, mf_d, 0, want_bits=False)
        torch.cuda.synchronize()
        k0.record()
        for _ in range(reps):
            rt.head_call(x0, mf_d, 0, want_bits=False)
        k1.record()
        torch.cuda.synchronize()
        kern_ms = kern_ms_burst = k0.elapsed_time(k1) / reps
        flops = einsum_flops_per_launch(Q, B)
        alg_bytes = B * C * (H // 4) * (W // 4) * 4 + B * Q * (H // 4) * (W // 4) * 4
        kname = 'cgg_head_call stage (fp32 SIMT heads + mask einsum of one head call)'
    # tensor roof: sustained loop against the sustained peak; HBM roof: the 10-launch timing against the copy peak (both
    # are burst measurements; MEASURED_PEAKS.json has no sustained HBM figure) -- the sustained-loop HBM fraction is
    # reported beside it
    ach_tf = flops / (kern_ms * 1e-3) / 1e12
    ach_gbs = alg_bytes / (kern_ms_burst * 1e-3) / 1e9
    ach_gbs_sus = alg_bytes / (kern_ms * 1e-3) / 1e9
    frac_t, frac_h = ach_tf / peaks['tflops'], ach_gbs / peaks['hbm_gbs']
    # the binding roof: arithmetic intensity against the ridge of the measured peaks
    ai, ridge = flops / alg_bytes, peaks['tflops'] * 1e12 / (peaks['hbm_gbs'] * 1e9)
    hbm_bound = ai < ridge
    traffic, traffic_src, write_only = None, None, None
    tpath = os.path.join(ROOT, 'profiles', 'einsum_dram_traffic.json')
    if args.precision == 'bf16' and os.path.exists(tpath):
        tj = json.load(open(tpath))
        if tj.get('batch') == B and tj.get('queries') == Q:
            traffic = tj.get('dram_bytes_per_launch')
            traffic_src = 'ncu --set full capture committed under profiles/ (%s); not re-measured in this run' % tj.get('source', '')
    wpath = os.path.join(ROOT, 'profiles', 'r02_hbm_write_ceiling.json')
    if os.path.exists(wpath):
        write_only = json.load(open(wpath))
    per_gpu_value = value / world
    trace('strong + roofline legs done')
    roofline = dict(bound='hbm' if hbm_bound else 'tensor',
                    achieved=ach_gbs if hbm_bound else ach_tf, peak=peaks['hbm_gbs'] if hbm_bound else peaks['tflops'],
                    unit='GB/s' if hbm_bound else 'TFLOP/s', frac=frac_h if hbm_bound else frac_t,
                    traffic=traffic, traffic_source=traffic_src, kernel=kname, kernel_ms=kern_ms_burst,
                    kernel_ms_sustained=kern_ms, launches_timed=[10, reps],
                    algorithmic_bytes=alg_bytes, algorithmic_flops=flops, arithmetic_intensity=ai, ridge=ridge,
                    tensor=dict(achieved=ach_tf, peak=peaks['tflops'], frac=frac_t, unit='TFLOP/s',
                                timing='>= 1 s back to back (sustained clocks) against the sustained bf16 peak',
                                frac_of_burst=flops / (kern_ms_burst * 1e-3) / 1e12 / peaks['tflops_burst']),
                    hbm=dict(achieved=ach_gbs, peak=peaks['hbm_gbs'], frac=frac_h, unit='GB/s',
                             timing='10 launches back to back against the copy peak (both burst-clock measurements)',
                             frac_sustained_clocks=ach_gbs_sus / peaks['hbm_gbs'],
                             write_only_ceiling=write_only),
                    peak_source=peaks['source'],
                    whole_path=dict(achieved=flops_per_image(Q) * per_gpu_value / 1e12, unit='TFLOP/s per GPU',
                                    frac=flops_per_image(Q) * per_gpu_value / 1e12 / peaks['tflops'],
                                    sustained_frac=flops_per_image(Q) * sustained['value'] / world / 1e12 / peaks['tflops']))

    # ---- stage / config legs
    grounding = train = matching_rec = pixdec = None
    if not args.no_train:
        try:
            # single-process stage legs: N = 1 only (the matching losses average their positives over the ranks -- a
            # collective -- so running them on rank 0 alone under torchrun would leave the other ranks out of step)
            grounding = grounding_leg(dev) if (rank == 0 and world == 1) else None
            matching_rec = matching_leg(dev) if (rank == 0 and world == 1) else None
            if rank == 0 and world == 1 and not args.no_pixel_decoder:
                try:
                    pixdec = pixel_decoder_leg(dev, B, heads[0])
                except Exception as e:      # noqa: BLE001
                    pixdec = dict(error=repr(e)[:300])
            del heads, fly_in
            torch.cuda.empty_cache()
            trace('stage legs done, train leg starts')
            train = train_leg(args, rank, world, dev)
            trace('train leg done')
        except Exception as e:      # noqa: BLE001
            train = dict(error=repr(e)[:300])
    tgb = None
    if rank == 0 and world == 1 and not args.no_torch_baseline:
        try:
            torch.cuda.empty_cache()
            tgb = torch_gpu_baseline(Q, B, dev)
            tgb['speedup_vs_faster'] = value / max(tgb['fp32'], tgb['bf16_autocast'])
        except Exception as e:      # noqa: BLE001
            tgb = dict(error=repr(e)[:300])

    if rank == 0:
        cpu = cpu_baseline(Q, os.cpu_count() or 1) if (world == 1 and not args.no_cpu_baseline) else None
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
                    ms_per_step=ms / args.steps, higher_is_better=True, scaling='weak', vs_baseline=None,
                    dtype='bf16' if args.precision == 'bf16' else 'f32', data='synthetic', impl='b200',
                    config=dict(workload='configs[1]: COCO-OVIS instance decoder head, Q=%d, 9 layers, 256-d, 8 heads, '
                                         '1024x1024, batch %d per GPU' % (Q, B),
                                batch_per_gpu=B, global_batch=B * world, precision=args.precision,
                                cuda_graph=not args.no_graph, in_flight_batches=n_fly,
                                final_mask_only=bool(args.final_mask_only),
                                single_batch_latency_ms=latency_ms,
                                single_batch_images_per_s=B / (latency_ms * 1e-3),
                                l2='inputs (%.0f MB per step) larger than L2, no explicit flush' % (h2d / 1e6),
                                flops_per_image=flops_per_image(Q), numa_pinned_cpus=numa_cpus),
                    e2e=dict(value=e2e_val, unit=UNIT, h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h, steps=e2e_steps),
                    gpu_launches=int(launches), roofline=roofline, clocks=clocks, sustained=sustained)
        if strong is not None:
            line['strong_scaling'] = strong
        if train is not None:
            line['train'] = train
        if grounding is not None:
            line['grounding'] = grounding
        if matching_rec is not None:
            line['matching_losses'] = matching_rec
        if pixdec is not None:
            line['pixel_decoder'] = pixdec
        if tgb is not None:
            line['torch_gpu_baseline'] = tgb
        if cpu is not None:
            line['cpu_baseline'] = cpu
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--batch', type=int, default=16, help='images per GPU per step')
    ap.add_argument('--precision', default='bf16', choices=['bf16', 'fp32'])
    ap.add_argument('--queries', type=int, default=100)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-torch-baseline', action='store_true')
    ap.add_argument('--no-train', action='store_true', help='skip the configs[3] training-step leg and the K7 stage leg')
    ap.add_argument('--no-pixel-decoder', action='store_true', help='skip the row-f3 pixel-decoder leg')
    ap.add_argument('--no-strong', action='store_true', help='skip the configs[2] strong-scaling leg')
    ap.add_argument('--train-batch', type=int, default=2, help='images per GPU in the training-step leg')
    ap.add_argument('--train-steps', type=int, default=5)
    ap.add_argument('--train-precision', choices=['fp32', 'tf32'], default='tf32',
                    help="arithmetic of the training step's contractions: tcgen05 kind::tf32 or fp32 FMA (parity mode)")
    ap.add_argument('--no-train-graph', action='store_true', help='time the training step eagerly only')
    ap.add_argument('--sustain-s', type=float, default=2.0, help='length of the sustained leg in seconds')
    ap.add_argument('--no-graph', action='store_true', help='launch the path eagerly instead of replaying a CUDA graph')
    ap.add_argument('--final-mask-only', action='store_true',
                    help='opt-in inference shortcut: produce the last head call mask only (NOT the headline contract)')
    ap.add_argument('--in-flight', type=int, default=4,
                    help='batches in flight in the device-resident throughput leg (one head + stream each)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one returned (rank 0) as DIR/<name>.npy, float32; '
                         'arrays too large for the %d MB budget as a fixed sample.  --impl b200 only: the reference '
                         'arm runs one image per step, not the b200 arm\'s batch, so its outputs would not line up'
                         % (DUMP_BYTES // 10**6))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs applies to --impl b200')
    if args.impl == 'reference':
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == '__main__':
    main()
