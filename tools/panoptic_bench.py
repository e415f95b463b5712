"""Fused panoptic output (postprocess.panoptic_postprocess_fused, cgg_panoptic_fuse) against the same step as plain
torch CUDA ops (oracle/panoptic_oracle.py on the GPU: what the reference executes -- full-resolution fp32 upsample of
every query, sigmoid, score product, argmax, and a Python loop over the kept queries with host syncs).

OSPS-shaped workloads (Q=200, 118 class rows, bf16 logits) at two planted kept-query counts each:
  B=1 at the reference's test shape: a 600x1000 image resized to 800x1333, padded to 800x1344, rescaled back;
  B=16 at 1024x1024 (no rescale).
Timing: CUDA events around each call, after a warm-up; a 512 MB buffer is overwritten between timed passes so that no
pass reads the logits from L2 (126 MB).  Prints one JSON line (and writes it to --out when given)."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from cgg_b200 import postprocess as P  # noqa: E402
from cgg_b200 import synth  # noqa: E402
from cgg_b200.head import build_head_from_state_dict  # noqa: E402
from oracle import panoptic_oracle as PO  # noqa: E402

Q, NCLS1, NUM_STUFF = 200, 118, 52        # 117 classes; the things / stuff split only decides which segments get ids
HBM_BPS = 7.7e12                          # HGX B200 data sheet, one GPU
MUFU_PER_CLK_SM, SMS = 16, 148            # sigmoid = ex2 + rcp on the MUFU pipe: 2 MUFU ops per evaluation


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader,nounits'],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, plim, clk = [x.strip() for x in q.split(',')]
    return dict(gpu=name, power_limit_w=float(plim), max_sm_clock_mhz=float(clk))


def make_case(B, lowres, kept, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    C = NCLS1 - 1
    probs = torch.full((B, Q, NCLS1), 0.1 / C, device=dev)
    probs[..., C] = 0.9                                             # void winners
    for b in range(B):
        ids = torch.randperm(Q, generator=g, device=dev)[:kept]
        labels = torch.randint(0, C, (kept,), generator=g, device=dev)
        sc = 0.82 + 0.17 * torch.rand(kept, generator=g, device=dev)
        probs[b, ids] = ((1 - sc) / C)[:, None].expand(kept, NCLS1).clone()
        probs[b, ids, labels] = sc
    h, w = lowres
    yy = torch.arange(h, device=dev, dtype=torch.float32)[:, None]
    xx = torch.arange(w, device=dev, dtype=torch.float32)[None, :]
    c = torch.rand((B, Q, 3), generator=g, device=dev)
    cy, cx = c[..., 0, None, None] * h, c[..., 1, None, None] * w
    r = 4.0 + c[..., 2, None, None] * h / 4
    logits = 6.0 * (1.0 - ((yy - cy) ** 2 + (xx - cx) ** 2) / r ** 2)
    logits = (logits + 0.5 * torch.randn(logits.shape, generator=g, device=dev)).to(torch.bfloat16)
    return probs, logits


def timed(fn, reps, flush):
    times = []
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    times.sort()
    return times[len(times) // 2]


def run(workload, B, metas, rescale, lowres, kept, head, reps, torch_reps, flush, info):
    dev = torch.device('cuda')
    probs, logits = make_case(B, lowres, kept, dev, seed=kept)
    fused = lambda: P.panoptic_postprocess_fused(head, probs, logits, metas, rescale=rescale)   # noqa: E731
    nt = head.num_things_classes

    def plain():
        return [PO.panoptic_from_lowres(probs[b], logits[b].float(), metas[b], nt, rescale)[0] for b in range(B)]

    for _ in range(3):
        fused()
    plain()
    torch.cuda.synchronize()
    t_fused = timed(fused, reps, flush)
    t_torch = timed(plain, torch_reps, flush)
    # agreement at the timed sizes: identical maps except pixels whose top-two score * sigmoid are within 4 fp32 ulps
    got = fused()
    bad = near_total = mism_total = pixels = 0
    for b in range(B):
        want, st = PO.panoptic_from_lowres(probs[b], logits[b].float(), metas[b], nt, rescale)
        pm = st['prob_masks']
        if pm.shape[0] >= 2:
            top = pm.topk(2, dim=0).values
            near = (top[0] - top[1]) <= 4 * torch.finfo(torch.float32).eps * top[0]
        else:
            near = torch.zeros_like(want, dtype=torch.bool)
        mism = got[b] != want
        bad += int((mism & ~near).sum())
        mism_total += int(mism.sum())
        near_total += int(near.sum())
        pixels += want.numel()
        del pm, st
    out_h, out_w = metas[0]['ori_shape'][:2] if rescale else metas[0]['img_shape'][:2]
    px = B * out_h * out_w
    kept_bytes = B * kept * lowres[0] * lowres[1] * 2 + px * 4 * 3       # kept bf16 planes + pan write, read, write
    evals = kept * px
    mufu_rate = MUFU_PER_CLK_SM * SMS * info['max_sm_clock_mhz'] * 1e6 / 2
    floor_bw, floor_sig = kept_bytes / HBM_BPS * 1e3, evals / mufu_rate * 1e3
    return dict(workload=workload, batch=B, kept_per_image=kept, out_hw=[out_h, out_w], lowres_hw=list(lowres),
                fused_ms=round(t_fused, 4), images_per_s=round(B / t_fused * 1e3, 1), torch_ms=round(t_torch, 3),
                speedup=round(t_torch / t_fused, 2),
                floor_ms=dict(hbm=round(floor_bw, 4), sigmoid_mufu=round(floor_sig, 4),
                              bound='sigmoid' if floor_sig > floor_bw else 'hbm'),
                check=dict(pixels=pixels, mismatched=mism_total, mismatched_outside_near_ties=bad, near_tie_pixels=near_total,
                           ok=bad == 0 and mism_total <= 1e-5 * pixels))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--torch-reps', type=int, default=3)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('panoptic_bench.py needs a CUDA device')
    info = gpu_info()
    dev = torch.device('cuda')
    sd = synth.make_params(seed=1, num_queries=Q, num_classes_p1=NCLS1)
    head = build_head_from_state_dict(sd, Q, NCLS1, 'bf16', dev, num_stuff_classes=NUM_STUFF)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    m1 = [dict(batch_input_shape=(800, 1344), img_shape=(800, 1333, 3), ori_shape=(600, 1000, 3))]
    m16 = [dict(batch_input_shape=(1024, 1024), img_shape=(1024, 1024, 3), ori_shape=(1024, 1024, 3))] * 16
    rows = []
    for kept in (10, 100):
        rows.append(run('B=1 800x1333 (padded 800x1344), rescale to 600x1000', 1, m1, True, (200, 336), kept, head, a.reps,
                        a.torch_reps, flush, info))
        rows.append(run('B=16 1024x1024', 16, m16, False, (256, 256), kept, head, a.reps, a.torch_reps, flush, info))
    line = json.dumps(dict(tool='panoptic_bench', **info, timing='CUDA events, median of %d fused / %d torch '
                           'passes after warm-up; 512 MB buffer overwritten between passes (L2 flushed)' % (a.reps, a.torch_reps),
                           q=Q, class_rows=NCLS1, num_stuff=NUM_STUFF, logits='bf16', results=rows))
    print(line)
    if a.out:
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
