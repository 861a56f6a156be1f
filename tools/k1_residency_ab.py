"""K1 forward alone on the DPO C2 tile (64 x 2048 x 128257 bf16 = 33.6 GB, far larger than the 126 MB L2), one
launch shape after another, round-robin over several rounds.

For each shape it reports the read rate (algorithmic bytes: every scored row read once) over >= 50 back-to-back
launches timed with CUDA events, the SM clock sampled by nvidia-smi during those launches, and -- from one launch
traced with torch.profiler -- the grid, the registers per thread, and the CTAs per SM launched and resident at
once.  It also checks that every shape returns the same log-probs and (max, logsum) bits as the first one.

    python tools/k1_residency_ab.py [--iters 60] [--rounds 3] [--shapes 70,30,0,70:32] [--out FILE.json]

Shapes are aa_logprob_set_tuning codes (see launch_fwd in csrc/logprob.cu), CODE:N with N CTAs per SM; 70 is the
persistent 16-CTAs/SM launch that the one-CTA-per-row default (0) replaced, 30 the same kernel on a resident-sized grid.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap = argparse.ArgumentParser()
ap.add_argument('--n', type=int, default=64, help='sequences (C2: 32 pairs)')
ap.add_argument('--L', type=int, default=2048)
ap.add_argument('--V', type=int, default=128257)
ap.add_argument('--shapes', default='70,30,0', help='tuning codes, each optionally CODE:CTAS_PER_SM')
ap.add_argument('--iters', type=int, default=60)
ap.add_argument('--rounds', type=int, default=3)
ap.add_argument('--out', default='')
a = ap.parse_args()
if a.iters < 50:
    ap.error('--iters below 50 does not measure a sustained rate')

import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from align_anything_b200 import _lib as Lb  # noqa: E402
from align_anything_b200 import ops  # noqa: E402

if not torch.cuda.is_available():
    raise SystemExit('k1_residency_ab: no CUDA device')
dev = 'cuda'
n, Lq, V = a.n, a.L, a.V
gen = torch.Generator(device=dev).manual_seed(0)
logits = torch.empty((n, Lq, V), dtype=torch.bfloat16, device=dev)
for i in range(n):
    logits[i] = (torch.randn((Lq, V), generator=gen, device=dev) * 2.5).bfloat16()
ids = torch.randint(2, V - 1, (n, Lq), generator=gen, device=dev)
lens = tuple([Lq] * n)
labels = ops.strip_pad_tail(ids, lens, V - 1, True)
plan = ops._dpo_plan(logits, lens, labels.stride(0))
lp = torch.zeros(plan.out_shape, dtype=torch.bfloat16, device=dev)
stat = torch.empty((2, plan.n_rows), dtype=torch.float32, device=dev)
read_bytes = plan.n_rows * V * 2
shapes = [x.strip() for x in a.shapes.split(',')]


def set_shape(code):
    v, _, c = code.partition(':')
    Lb.check(Lb.lib().aa_logprob_set_tuning(int(v), int(c or 0)))


def fwd():
    ops._launch_fwd(logits, labels, plan, lp, stat[0], stat[1])


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip()


def timed(iters):
    """ms per launch over `iters` back-to-back launches, and the median SM clock sampled meanwhile."""
    smi = subprocess.Popen(['nvidia-smi', '--query-gpu=clocks.sm', '--format=csv,noheader,nounits', '-lms', '50'],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    try:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fwd()
        e1.record()
        torch.cuda.synchronize()
    finally:
        time.sleep(0.06)
        smi.terminate()
        out, _ = smi.communicate(timeout=10)
    mhz = [float(x) for x in out.split() if x.replace('.', '', 1).isdigit()]
    return e0.elapsed_time(e1) / iters, (statistics.median(mhz) if mhz else None)


def launch_shape():
    """grid, block, registers and resident CTAs per SM of one traced launch."""
    with tempfile.TemporaryDirectory() as td:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fwd()
            torch.cuda.synchronize()
        path = os.path.join(td, 'trace.json')
        prof.export_chrome_trace(path)
        ev = [e for e in json.load(open(path))['traceEvents']
              if e.get('cat') == 'kernel' and 'logprob_fwd' in e.get('name', '')]
    if not ev:
        return {}
    g = ev[0]['args']
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    grid, threads, regs = g['grid'][0], g['block'][0], g['registers per thread']
    # register file: 64 K per SM, allocated per warp in 256-register units; at most 64 warps and 32 CTAs per SM
    warps = -(-threads // 32)
    per_warp = -(-regs * 32 // 256) * 256
    resident = min(65536 // per_warp // warps, 64 // warps, 32)
    return {'kernel': ev[0]['name'], 'grid': grid, 'threads': threads, 'registers': regs,
            'launched_ctas_per_sm': round(grid / sms, 2), 'resident_ctas_per_sm': resident}


result = {'gpu': gpu_info(), 'tile': f'{n} x {Lq} x {V} bf16, {plan.n_rows} scored rows',
          'read_bytes_per_launch': read_bytes, 'iters_per_sample': a.iters, 'rounds': a.rounds, 'shapes': {}}
ref = None
for code in shapes:
    set_shape(code)
    for _ in range(3):  # warm-up
        fwd()
    torch.cuda.synchronize()
    out = (lp.clone(), stat.clone())
    if ref is None:
        ref = out
    same = bool(torch.equal(out[0].view(torch.int16), ref[0].view(torch.int16))
                and torch.equal(out[1].view(torch.int32), ref[1].view(torch.int32)))
    n_diff = int((out[1].view(torch.int32) != ref[1].view(torch.int32)).sum() +
                 (out[0].view(torch.int16) != ref[0].view(torch.int16)).sum())
    result['shapes'][code] = dict(launch_shape(), bit_identical_to_first=same, differing_elements=n_diff, ms=[],
                                  sm_mhz=[])
for r in range(a.rounds):
    for code in shapes:
        set_shape(code)
        fwd()
        torch.cuda.synchronize()
        ms, mhz = timed(a.iters)
        result['shapes'][code]['ms'].append(round(ms, 4))
        result['shapes'][code]['sm_mhz'].append(mhz)
        print(f'round {r} shape {code:>5s}: {ms:.3f} ms  {read_bytes / ms / 1e9:.3f} TB/s  SM {mhz} MHz', flush=True)
set_shape('0')
for code, s in result['shapes'].items():
    med = statistics.median(s['ms'])
    s['ms_median'] = med
    s['tbs_median'] = round(read_bytes / med / 1e9, 3)
    s['ms_spread'] = round(max(s['ms']) - min(s['ms']), 4)
print(json.dumps(result, indent=1))
if a.out:
    with open(a.out, 'w') as f:
        json.dump(result, f, indent=1)
