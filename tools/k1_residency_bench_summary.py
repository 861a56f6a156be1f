"""Summarise alternating bench.py runs of the old K1 launch (bench_old_<i>.json, --variant 70) and the default
(bench_new_<i>.json) in one directory: the median and spread of every headline number per arm, and new / old.

    python tools/k1_residency_bench_summary.py DIR
"""
import glob
import json
import os
import statistics
import sys


def last_json(path):
    for line in reversed(open(path).read().splitlines()):
        try:
            return json.loads(line)
        except ValueError:
            continue
    return None


METRICS = {
    'C2 value (pairs/s)': lambda d: d['value'],
    'C2 k1_fwd ms': lambda d: d['kernel_ms']['k1_fwd'],
    'C2 k1b_bwd ms': lambda d: d['kernel_ms']['k1b_bwd'],
    'C2 SM MHz': lambda d: d['clocks']['sm_mhz'],
    'C3 value': lambda d: d['other_configs']['C3']['value'],
    'C3 k1_fwd ms': lambda d: d['other_configs']['C3']['kernel_ms']['k1_fwd'],
    'C5 value': lambda d: d['other_configs']['C5']['value'],
    'C5 k1_fwd ms': lambda d: d['other_configs']['C5']['kernel_ms']['k1_fwd'],
    'ppo value (tokens/s)': lambda d: d['ppo']['value'],
    'ragged value (pairs/s)': lambda d: d['ragged']['value'],
    'sft_cross_entropy single_pass ms': lambda d: d['sft_cross_entropy']['single_pass']['ms'],
}

out = sys.argv[1]
arms = {}
for arm in ('old', 'new'):
    runs = [last_json(p) for p in sorted(glob.glob(os.path.join(out, f'bench_{arm}_*.json')))]
    arms[arm] = [r for r in runs if r]
for name, get in METRICS.items():
    row = []
    med = {}
    for arm in ('old', 'new'):
        vals = []
        for r in arms[arm]:
            try:
                vals.append(float(get(r)))
            except (KeyError, TypeError, ValueError):
                pass
        if vals:
            med[arm] = statistics.median(vals)
            row.append(f'{arm} {med[arm]:.4g} (spread {max(vals) - min(vals):.3g}, n={len(vals)})')
        else:
            row.append(f'{arm} -')
    ratio = f'new/old {med["new"] / med["old"]:.4f}' if len(med) == 2 and med['old'] else ''
    print(f'{name:34s} ' + '   '.join(row) + f'   {ratio}')
