"""The matching-based losses of one training step on panoptic ground truth as mmdet's data pipeline hands it over
(BitmapMasks at image size, a uint8 semantic map padded with 255), at the OSPS training shapes of BASELINE.json configs[3]:
B=2, Q=200, 118 class rows (64 things + 53 stuff: 117 = 64 + COCO's 53 stuff classes, the p20 config itself is not in
this tree), 1024^2 padded input, 256^2 mask logits, 15 thing masks and 10 stuff segments per image, 12 544 points.
One step = target preparation + `loss_single` of all 10 head calls, forward and backward (mask / class logits are leaf
tensors, the decoder itself is not run).  Paths:
  dense    the oracle's preprocess_gt (oracle/panoptic_targets_oracle.py) run on the device -- padded int64 masks, the
           reference's format -- then MatchingLosses on those dense masks;
  compact  head.preprocess_gt (cgg_b200/matching.py: stuff labels on the device, unpadded uint8 things planes) then
           MatchingLosses on the compact targets.
Reports the GPU name and power limit, the median wall time per step over --steps steps after --warmup (host clock around
a step that ends in a device synchronise), torch.cuda.max_memory_allocated per path, and whether both paths give equal
loss dicts on the same seeded CPU point draws.  One JSON line, also written to --out."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

NT, NS, Q, B, CALLS = 64, 53, 200, 2, 10
PAD, H4 = 1024, 256


class Bitmap:
    """The part of mmdet's BitmapMasks that preprocess_gt reads."""

    def __init__(self, masks):
        self.masks = masks
        self.height, self.width = masks.shape[1:]


def make_gt(seed):
    g = np.random.default_rng(seed)
    labels, masks, metas = [], [], []
    sem = np.full((B, 1, PAD, PAD), 255, np.uint8)
    for b in range(B):
        h, w = PAD - 24 - 40 * b, PAD - 8 - 16 * b                     # image size inside the padded input
        yy, xx = np.mgrid[:h, :w]
        m = np.zeros((15, h, w), np.uint8)
        for k in range(15):                                            # ellipses of varying size
            cy, cx = g.uniform(0.1, 0.9) * h, g.uniform(0.1, 0.9) * w
            ry, rx = g.uniform(0.03, 0.25) * h, g.uniform(0.03, 0.25) * w
            m[k] = ((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1
        lab = g.integers(0, NT, 15)
        s = np.full((h, w), 255, np.uint8)
        for k, sl in enumerate(g.choice(NS, 10, replace=False)):       # 10 stuff bands
            s[k * h // 10:(k + 1) * h // 10] = NT + sl
        for k in range(15):
            s[m[k] > 0] = lab[k]                                       # thing pixels carry thing labels
        sem[b, 0, :h, :w] = s
        labels.append(torch.from_numpy(lab).long())
        masks.append(Bitmap(m))
        metas.append(dict(pad_shape=(PAD, PAD, 3)))
    return labels, masks, torch.from_numpy(sem), metas


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader,nounits'],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, plim, clk = [x.strip() for x in q.split(',')]
    return dict(gpu=name, power_limit_w=float(plim), max_sm_clock_mhz=float(clk))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=7)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    from cgg_b200 import matching
    from oracle import panoptic_targets_oracle as PT
    assert torch.cuda.is_available(), 'this benchmark measures the GPU'
    dev = torch.device('cuda', 0)
    labels, bitmaps, sem, metas = make_gt(0)
    g = torch.Generator().manual_seed(1)
    mask_preds = [(torch.randn((B, Q, H4, H4), generator=g) * 2).to(dev).requires_grad_(True) for _ in range(CALLS)]
    cls = [torch.randn((B, Q, NT + NS + 1), generator=g).to(dev).requires_grad_(True) for _ in range(CALLS)]
    emb = [(torch.randn((B, Q, NT + NS + 1), generator=g) * 2).to(dev).requires_grad_(True) for _ in range(CALLS)]
    ml = matching.MatchingLosses(types.SimpleNamespace(num_classes=NT + NS))

    def dense_targets():
        mm = [torch.from_numpy(m.masks).to(dev) for m in bitmaps]
        lab, masks = PT.preprocess_gt([x.to(dev) for x in labels], mm, sem.to(dev), metas, NT, NS)
        return lab, masks

    def compact_targets():
        return matching.preprocess_gt(labels, bitmaps, sem.to(dev), metas, NT, NS, dev)

    def step(prep):
        for t in mask_preds + cls + emb:
            t.grad = None
        lab, tg = prep()
        total, out = 0.0, {}
        for j in range(CALLS):
            o, _, _ = ml.loss_single(cls[j], emb[j], mask_preds[j], lab, tg)
            total = total + sum(o.values())
            out.update({'d%d.%s' % (j, k): v.detach() for k, v in o.items()})
        total.backward()
        return out

    paths = dict(dense=dense_targets, compact=compact_targets)
    # equality on the same seeded CPU point draws
    ml.rand = lambda *shape, device=None: torch.rand(*shape)
    ref = {}
    for name, prep in paths.items():
        torch.manual_seed(5)
        ref[name] = {k: v.cpu() for k, v in step(prep).items()}
    equal = all(torch.equal(ref['dense'][k], ref['compact'][k]) for k in ref['dense'])
    ml.rand = lambda *shape, device=None: torch.rand(*shape, device=device)     # the product's draws, on the device
    res = dict(gpu_info(), workload=dict(B=B, Q=Q, things=NT, stuff=NS, pad=PAD, logits=H4, thing_masks=15,
                                         stuff_segments=10, head_calls=CALLS, num_points=ml.num_points),
               losses_equal=equal, steps=args.steps, warmup=args.warmup)
    times = {k: [] for k in paths}
    peak = {}
    for name, prep in paths.items():
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        for _ in range(args.warmup):
            step(prep)
        torch.cuda.synchronize()
        peak[name] = (torch.cuda.max_memory_allocated() - base) / 2 ** 20
    for _ in range(args.steps):                                                  # alternate the two paths
        for name, prep in paths.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            step(prep)
            torch.cuda.synchronize()
            times[name].append((time.perf_counter() - t0) * 1e3)
    for name in paths:
        res[name] = dict(median_ms=round(statistics.median(times[name]), 3), min_ms=round(min(times[name]), 3),
                         max_ms=round(max(times[name]), 3), peak_mib_above_inputs=round(peak[name], 1))
    res['speedup'] = round(res['dense']['median_ms'] / res['compact']['median_ms'], 3)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
