"""The bf16 GEMM stages at shapes other than the benchmark's: 1056x800 and 768^2 with Q=100 (odd pixel / key tile
counts), 1024^2 with Q=128 and Q=240 (the pixel-on-lane pair einsum, one and two N tiles per head call) and Q=300
(also two attention-mask query slices).  Per shape it times the CUDA-graph decoder forward at B=16, cgg_kv_project
and the 10-call cgg_mask_einsum (CUDA events, median of 5 windows of --iters back-to-back calls) and prints one JSON
line with the GPU's name and power limit.  With --dump DIR it also writes the masks, the attention-mask bitmaps and
the K/V buffers of one seeded eager B=1 forward per shape; --compare A B prints, per shape and output, the largest
difference between two such dumps.  --root is the repository whose package is imported, so that one copy of this
script measures two trees; --queries restricts the run to shapes with those query counts.
Usage: python tools/gemm_routes_bench.py [--root DIR] [--iters N] [--dump DIR] [--queries 100,300]
       python tools/gemm_routes_bench.py --compare DIR_A DIR_B"""
import argparse
import json
import os
import subprocess
import sys

SHAPES = [(100, 1056, 800), (100, 768, 768), (128, 1024, 1024), (240, 1024, 1024), (300, 1024, 1024)]


def gpu_name(torch):
    try:
        return subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                              capture_output=True, text=True).stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        return torch.cuda.get_device_name(0)


def median_ms(torch, fn, iters, windows=5):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = []
    for _ in range(windows):
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b) / iters)
    return sorted(out)[windows // 2]


def run(args):
    sys.path.insert(0, os.path.abspath(args.root))
    import torch
    from cgg_b200 import synth
    from cgg_b200.head import build_head_from_state_dict
    dev = torch.device('cuda', 0)
    gpu = gpu_name(torch)
    for Q, H, W in SHAPES:
        if args.queries and Q not in args.queries:
            continue
        sd = synth.make_params(seed=0, num_queries=Q)
        mf, mems = synth.make_inputs(0, 16, H, W, dtype=torch.bfloat16)
        mf, mems = mf.to(dev), [m.to(dev) for m in mems]
        head = build_head_from_state_dict(sd, Q, 49, 'bf16', dev, cuda_graph=True)
        fwd = median_ms(torch, lambda: head.decoder_forward(mf, mems), args.iters)
        rt = head._runtime(dev)
        kv = median_ms(torch, lambda: rt.kv_project(mems), args.iters)
        out = torch.empty((10,) + (16, Q) + tuple(mf.shape[-2:]), dtype=torch.bfloat16, device=dev)
        ein = median_ms(torch, lambda: rt.mask_einsum(mf, out), args.iters)
        print(json.dumps(dict(root=args.root, Q=Q, H=H, W=W, B=16, forward_graph_ms=round(fwd, 4),
                              kv_project_ms=round(kv, 4), mask_einsum_10_calls_ms=round(ein, 4), gpu=gpu)), flush=True)
        del head, rt, out
        torch.cuda.empty_cache()
        if args.dump:
            head = build_head_from_state_dict(sd, Q, 49, 'bf16', dev)
            cls, emb, mask, dbg = head.decoder_forward(mf[:1].contiguous(), [m[:1].contiguous() for m in mems],
                                                       return_debug=True)
            rt = head._runtime(dev)
            torch.cuda.synchronize()
            kv = []
            for lvl, m in enumerate(mems):      # (1, K_l, nl * 2C) bf16, nl = layers reading level l
                off = rt.lib.cgg_workspace_offset(rt.handle, 1, b'kv%d' % lvl)
                n = m.shape[-2] * m.shape[-1] * len(range(lvl, head.num_transformer_decoder_layers, 3)) * 2 * 256
                kv.append(rt.workspace[off:off + 2 * n].view(torch.bfloat16).cpu())
            os.makedirs(args.dump, exist_ok=True)
            torch.save(dict(mask=[m.cpu() for m in mask], bits=[b.cpu() for b in dbg['bitmaps']], kv=kv),
                       os.path.join(args.dump, 'q%d_%dx%d.pt' % (Q, H, W)))
            del head, rt
            torch.cuda.empty_cache()


def compare(a, b):
    import torch
    for Q, H, W in SHAPES:
        name = 'q%d_%dx%d.pt' % (Q, H, W)
        if not (os.path.exists(os.path.join(a, name)) and os.path.exists(os.path.join(b, name))):
            continue
        x, y = torch.load(os.path.join(a, name)), torch.load(os.path.join(b, name))
        res = dict(Q=Q, H=H, W=W)
        for j, (m, n) in enumerate(zip(x['mask'], y['mask'])):
            d = float((m.float() - n.float()).abs().max()) / float(m.float().abs().max())
            res['mask%d' % j] = 0.0 if torch.equal(m, n) else d
        res['bit_words_differing'] = [int((p != q).sum()) for p, q in zip(x['bits'], y['bits'])]
        res['kv'] = [0.0 if torch.equal(p, q) else float((p.float() - q.float()).abs().max()) / float(p.float().abs().max())
                     for p, q in zip(x['kv'], y['kv'])]
        print(json.dumps(res), flush=True)


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--root', default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--dump', default=None)
    ap.add_argument('--compare', nargs=2, default=None)
    ap.add_argument('--queries', type=lambda s: [int(q) for q in s.split(',')], default=None)
    args = ap.parse_args()
    if args.compare:
        compare(*args.compare)
    else:
        run(args)
