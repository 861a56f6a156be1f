"""The SFT / PTX cross-entropy with and without the (B, L, V) logits tile, forward + backward down to d(hidden) and
d(weight), on one GPU.  Prints one JSON line.

    python tools/sft_fused_lm_head.py [--reps 5] [--warmup 2] [--shapes 128256x4096,128257x4096,152064x3584]

Batch: 8 x 2048 positions, prompts masked as in bench.sft_ce_bench (prompt length uniform in [L/8, L/2), labels -100).
Arms, each timed from the last hidden states and the lm_head weight to both gradients:
  fused        ops.causal_lm_loss_from_hidden: aa_ce_rows, the valid rows gathered, K6 forward, K6b + aa_linear_dhidden +
               aa_linear_dweight backward (4 GEMM passes over the valid rows, tcgen05)
  materialised F.linear (cuBLAS) + ops.causal_lm_loss (K1f): logits and gradient tiles over every position
  eager        F.linear + F.cross_entropy(logits.float()): transformers' ForCausalLMLoss arithmetic on ATen
Per arm: median ms over CUDA events (one forward + backward each, synchronised), the peak memory allocated beyond what
was live before the call (inputs, weights; the gradients it produces count), the loss, and TFLOP/s over the fused
path's 4 GEMM passes (4 * 2 * n_valid * H * V flops / ms, the same numerator for every arm).  The device name, power
limit and max SM clock are read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SAMPLES, SEQ = 8, 2048


def device_facts():
    facts = {'device': torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        p, c = (x.strip() for x in r.stdout.strip().split(','))
        facts.update(power_limit=p, sm_clock_max=c)
    except Exception as e:  # the numbers still stand; say that the limit could not be read
        facts['power_limit'] = f'not read ({type(e).__name__})'
    return facts


def batch(V, H, device):
    gen = torch.Generator().manual_seed(3)  # bench.sft_ce_bench's masking
    labels = torch.randint(0, V, (SAMPLES, SEQ), generator=gen)
    prompt = torch.randint(SEQ // 8, SEQ // 2, (SAMPLES,), generator=gen)
    for b in range(SAMPLES):
        labels[b, : int(prompt[b])] = -100
    g = torch.Generator(device=device).manual_seed(11)
    hidden = torch.randn((SAMPLES, SEQ, H), generator=g, device=device).bfloat16()
    weight = (torch.randn((V, H), generator=g, device=device) * 0.02).bfloat16()
    return hidden, weight, labels.to(device)


def arm_fn(name, ops):
    if name == 'fused':
        return lambda h, w, y: ops.causal_lm_loss_from_hidden(h, w, y)
    if name == 'materialised':
        return lambda h, w, y: ops.causal_lm_loss(F.linear(h, w), y)

    def eager(h, w, y):
        logits = F.linear(h, w).float()
        shift = F.pad(y, (0, 1), value=-100)[..., 1:]
        return F.cross_entropy(logits.view(-1, logits.size(-1)), shift.reshape(-1), ignore_index=-100)

    return eager


def measure(fn, h, w, y, reps, warmup, device):
    ts, peaks, loss = [], [], None
    for r in range(warmup + reps):
        h.grad = w.grad = None
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(device)
        base = torch.cuda.memory_allocated(device)
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        out = fn(h, w, y)
        out.backward()
        t1.record()
        torch.cuda.synchronize()
        if r >= warmup:
            ts.append(t0.elapsed_time(t1))
            peaks.append(torch.cuda.max_memory_allocated(device) - base)
        loss = float(out.detach())
        del out
    return {'ms': statistics.median(ts), 'ms_min': min(ts), 'ms_max': max(ts), 'peak_extra_gb': max(peaks) / 1e9,
            'loss': loss}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--shapes', default='128256x4096,128257x4096,152064x3584', help='VxH,...')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('sft_fused_lm_head.py measures on a GPU; none is visible')
    from align_anything_b200 import ops

    device = torch.device('cuda', 0)
    torch.cuda.set_device(device)
    result = {'metric': 'SFT cross-entropy forward + backward to d(hidden), d(weight)', **device_facts(),
              'batch': {'samples': SAMPLES, 'seq_len': SEQ}, 'reps': args.reps, 'warmup': args.warmup,
              'memory_note': 'peak_extra_gb = max_memory_allocated - memory_allocated before the call (the produced '
                             'gradients included)', 'shapes': []}
    for spec in args.shapes.split(','):
        V, H = (int(x) for x in spec.lower().split('x'))
        hidden, weight, labels = batch(V, H, device)
        n_valid = int((labels[:, 1:] != -100).sum())
        h, w = hidden.requires_grad_(True), weight.requires_grad_(True)
        flops4 = 4 * 2 * n_valid * H * V
        row = {'V': V, 'H': H, 'valid_rows': n_valid, 'positions': SAMPLES * SEQ,
               'fused_gemm_tflop': flops4 / 1e12, 'materialised_gemm_tflop': 3 * 2 * SAMPLES * SEQ * H * V / 1e12}
        for name in ('fused', 'materialised', 'eager'):
            m = measure(arm_fn(name, ops), h, w, labels, args.reps, args.warmup, device)
            m['tflops_over_fused_4_passes'] = flops4 / m['ms'] / 1e9
            row[name] = m
            torch.cuda.empty_cache()
        ops.check_status(device)
        f, mat = row['fused'], row['materialised']
        row['fused_vs_materialised'] = {
            'speedup': mat['ms'] / f['ms'], 'memory_saved_gb': mat['peak_extra_gb'] - f['peak_extra_gb'],
            'memory_ratio': f['peak_extra_gb'] / mat['peak_extra_gb'],
            'loss_rel_diff': abs(f['loss'] - mat['loss']) / abs(mat['loss']),
            'loss_rel_diff_vs_eager': abs(f['loss'] - row['eager']['loss']) / abs(row['eager']['loss'])}
        result['shapes'].append(row)
        del hidden, weight, h, w, labels
        torch.cuda.empty_cache()
    print(json.dumps(result))


if __name__ == '__main__':
    main()
