"""Device time of the masked cross-attention kernel inside real eager B=16 1024^2 Q=100 bf16 forwards, grouped by key
count (torch.profiler with CUDA activities).  Layer j's cross-attention attends to the keys of level j % 3; each layer
also runs the Q x Q self-attention on the same kernel.  The helper kernel that computes the live-tile flags is
reported on its own line.  Prints JSON lines; with an output path, also writes them there.
Usage: python tools/attention_profile.py [forwards] [output.jsonl]"""
import json, os, re, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from torch.profiler import profile, ProfilerActivity
from cgg_b200 import synth
from cgg_b200.head import build_head_from_state_dict

B, Q, SIZE = 16, 100, 1024
N_FWD = int(sys.argv[1]) if len(sys.argv) > 1 else 5
ATTN = re.compile(r'masked_attention_tc_kernel|attention_tc3_kernel')   # this tree's kernel / the earlier name
LIVE = re.compile(r'attention_live_kernel')

dev = torch.device('cuda', 0)
sd = synth.make_params(seed=0, num_queries=Q)
head = build_head_from_state_dict(sd, Q, 49, 'bf16', dev)
mf, mems = synth.make_inputs(0, B, SIZE, SIZE, dtype=torch.bfloat16)
mf, mems = mf.to(dev), [m.to(dev) for m in mems]
level_keys = [int(m.shape[-2] * m.shape[-1]) for m in mems]
for _ in range(3):
    head.decoder_forward(mf, mems)
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(N_FWD):
        head.decoder_forward(mf, mems)
    torch.cuda.synchronize()

evs = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA), key=lambda e: e.time_range.start)
attn = [e for e in evs if ATTN.search(e.name)]
live = [e for e in evs if LIVE.search(e.name)]
per_fwd = len(attn) // N_FWD
assert per_fwd * N_FWD == len(attn) and per_fwd % 2 == 0, (len(attn), N_FWD)
groups = {}
for i, e in enumerate(attn):
    j, cross = divmod(i % per_fwd, 2)
    keys = level_keys[j % len(level_keys)] if cross == 0 else Q
    groups.setdefault((keys, 'cross' if cross == 0 else 'self'), []).append(e.time_range.elapsed_us())

try:
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
except (OSError, IndexError):
    gpu = torch.cuda.get_device_name(0)
out_path = sys.argv[2] if len(sys.argv) > 2 else None
with open(out_path, 'w') if out_path else open(os.devnull, 'w') as f:
    def emit(**kw):
        line = json.dumps(kw)
        print(line, flush=True)
        f.write(line + '\n')
    kernel = attn[0].name if attn else None
    total = sum(sum(v) for v in groups.values()) / N_FWD
    for (keys, kind), us in sorted(groups.items()):
        us = sorted(us)
        emit(kernel=kernel, kind=kind, keys=keys, launches_per_forward=len(us) // N_FWD, median_us=us[len(us) // 2],
             min_us=us[0], max_us=us[-1], gpu=gpu)
    if live:
        us = sorted(e.time_range.elapsed_us() for e in live)
        emit(kernel=live[0].name, kind='live_flags', launches_per_forward=len(us) // N_FWD, median_us=us[len(us) // 2],
             min_us=us[0], max_us=us[-1], gpu=gpu)
        total += sum(us) / N_FWD
    emit(kind='per_forward_total', attention_us=total, batch=B, size=SIZE, Q=Q, forwards=N_FWD, gpu=gpu)
