"""Caption generation at test time (simple_test(with_caption=True), inference.py:84-157) on the real caption transformer
(4 blocks, 768, FFN 512, 8 heads, 30 522 tokens, Q=100 query embeddings), seeded weights with the [SEP] bias lifted so
that caption lengths vary from image to image.  Workloads: B=1 and B=16 images.  Arms, each timed per batch and per image:
  product    a tree's search: `beam_search_batch` (every image at once on the device) when the tree has it, otherwise the
             per-image `beam_search` (host loop, one blocking copy per step);
  reference  the oracle's beam search (oracle/caption_oracle.py) as plain torch CUDA ops, one image at a time, with its
             id tensors created on the GPU.
With --parent DIR (a checkout of another tree, built), the product of this tree and of DIR are measured in alternating
worker processes, `--rounds` times each, so that a clock or power drift during the run falls on both; the reference is
measured in this tree's workers.  Every arm's time is the median over all its repetitions (host clock around a call that
ends in a device synchronise, after one warm-up call per workload; the weights, ~140 MB, stay L2 / HBM resident across
calls as in an evaluation loop).  Checks that every arm gives the same ids and finished sequences for every image.  Prints
one JSON line and writes it to --out."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CFG = dict(nb_layers=4, input_dim=768, hidden_dim=768, ff_dim=512, nb_heads=8, drop_val=0.0, pre_norm=False, seq_length=35,
           nb_tokens=30522)
BOS, EOS, Q = 101, 102, 100


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader,nounits'],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, plim, clk = [x.strip() for x in q.split(',')]
    return dict(gpu=name, power_limit_w=float(plim), max_sm_clock_mhz=float(clk))


def worker(tree, reps, eos_bias, with_reference):
    """One process, one tree: per workload the product's times, steps and results (and the reference's)."""
    sys.path.insert(0, ROOT)
    sys.path.insert(0, tree)                  # the tree's package first; the oracle is this tree's
    import torch
    from cgg_b200 import caption, synth
    from cgg_b200.head import Mask2FormerHeadOpenB200
    from oracle import caption_oracle as CO

    class DeviceIds:
        """`torch` as the oracle sees it, with torch.tensor creating its id / weight tensors on the memory's device."""

        def __init__(self, dev):
            self.dev = dev

        def __getattr__(self, name):
            return getattr(torch, name)

        def tensor(self, data, **kw):
            if isinstance(data, list) and data and torch.is_tensor(data[0]):
                data = [float(x) for x in data]
            return torch.tensor(data, device=self.dev, **kw)

    def reference(sd, memory):
        out = []
        orig = CO.torch
        CO.torch = DeviceIds(memory.device)
        try:
            for b in range(memory.shape[0]):
                best, finished = CO.beam_search(sd, CFG, memory[b:b + 1], BOS, EOS)
                out.append([best, [f[0] for f in finished]])
        finally:
            CO.torch = orig
        return out

    def product(head, memory):
        if hasattr(caption, 'beam_search_batch'):
            res = caption.beam_search_batch(head, memory)
        else:
            res = [caption.beam_search(head, memory[b:b + 1]) for b in range(memory.shape[0])]
        return [[r['ids'], [f[0] for f in r['finished']]] for r in res]

    def timed(fn):
        ts = []
        for _ in range(reps):
            torch.cuda.synchronize()
            t = time.perf_counter()
            r = fn()
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t) * 1e3)
        return r, ts

    dev = torch.device('cuda')
    sd = synth.make_caption_params(3, cfg=CFG, eos_bias=eos_bias)
    head = Mask2FormerHeadOpenB200(num_things_classes=48, num_stuff_classes=0, num_queries=Q, use_class_emb=True,
                                   use_caption=True, use_caption_generation=True, bert_vocab_size=CFG['nb_tokens'],
                                   caption_generator=dict(type='CaptionTransformer', **CFG))
    head.load_state_dict(sd, strict=False)
    head = head.to(dev).eval()
    sd = {k: v.to(dev) for k, v in sd.items()}
    sd['caption_generator.position_encoder.psne_layer'] = CO.positions(35, 768).to(dev)
    memory = torch.randn((16, Q, 768), generator=torch.Generator().manual_seed(17)).to(dev)
    impl = 'batched' if hasattr(caption, 'beam_search_batch') else 'per_image'
    out = dict(impl=impl, workloads={})
    for B in (1, 16):
        mem = memory[:B].contiguous()
        with torch.no_grad():
            product(head, mem)                                                   # warm-up
            got, ms = timed(lambda: product(head, mem))
            w = dict(product_ms=ms, results=got, steps=None)
            if impl == 'batched':
                st, w['steps'] = caption._search_device(head, mem, BOS, EOS, 35, 7, 0.7)
                caption._search_results(st)
            if with_reference:
                reference(sd, mem[:1])                                           # warm-up
                w['reference'], w['reference_ms'] = timed(lambda: reference(sd, mem))
        out['workloads'][B] = w
    return out


def run_worker(tree, args, with_reference):
    cmd = [sys.executable, os.path.abspath(__file__), '--worker', tree, '--reps', str(args.reps), '--eos-bias',
           str(args.eos_bias)] + (['--with-reference'] if with_reference else [])
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise SystemExit('worker failed on %s' % tree)
    return json.loads(r.stdout.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--parent', default=None, help='another tree (built) whose search is timed alternately with this one')
    ap.add_argument('--eos-bias', type=float, default=2.5)
    ap.add_argument('--reps', type=int, default=3, help='repetitions per arm and workload in each worker')
    ap.add_argument('--rounds', type=int, default=2, help='worker processes per tree, alternating')
    ap.add_argument('--worker', default=None, help=argparse.SUPPRESS)
    ap.add_argument('--with-reference', action='store_true', help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        print(json.dumps(worker(args.worker, args.reps, args.eos_bias, args.with_reference)))
        return
    trees = [('this', ROOT)] + ([('parent', os.path.abspath(args.parent))] if args.parent else [])
    runs = {name: [] for name, _ in trees}
    for rnd in range(args.rounds):
        for name, tree in (trees if rnd % 2 == 0 else trees[::-1]):
            runs[name].append(run_worker(tree, args, with_reference=(name == 'this')))
    line = dict(bench='caption_beam_search', eos_bias=args.eos_bias, reps=args.reps, rounds=args.rounds, **gpu_info(),
                impl={name: runs[name][0]['impl'] for name in runs}, workloads=[])
    for B in ('1', '16'):
        this = [r['workloads'][B] for r in runs['this']]
        want = this[0]['reference']
        lengths = [len(ids) for ids, _ in want if ids is not None]
        w = dict(B=int(B), mean_caption_length=sum(lengths) / max(1, len(lengths)), captions_found=len(lengths))
        for name in runs:
            ws = [r['workloads'][B] for r in runs[name]]
            ms = statistics.median([t for x in ws for t in x['product_ms']])
            w[name] = dict(ms_per_batch=ms, ms_per_image=ms / int(B), steps_issued=ws[0]['steps'],
                           matches_reference=all(x['results'] == want for x in ws))
        ms = statistics.median([t for x in this for t in x['reference_ms']])
        w['reference'] = dict(ms_per_batch=ms, ms_per_image=ms / int(B),
                              deterministic=all(x['reference'] == want for x in this))
        line['workloads'].append(w)
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(s + '\n')


if __name__ == '__main__':
    main()
