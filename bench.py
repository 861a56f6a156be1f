#!/usr/bin/env python
"""bench.py -- RLHF loss hot path on B200: preference-pairs/s (DPO) and scored rollout-tokens/s (PPO) on synthetic
batches shaped like BASELINE.json's configs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config C2|C3|C4|C5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

    C2 (default, the headline): Llama-3-8B shapes text->text DPO, V = 128257, seq_len 2048, 32 pairs/step, bf16
    C3: LLaVA-1.5-7B shapes text+image->text DPO, V = 32064, seq_len 2048, 576 image positions in the prompt
    C4: Qwen2-VL-7B shapes text+image->text PPO (actor + critic + RM), V = 152064, H = 3584, 512-token responses
    C5: Qwen2-Audio-7B shapes text+audio->text DPO, V = 156032, seq_len 4096, 750 audio positions in the prompt
    (C1, OPT-125M on CPU, is the reference's own plumbing case: tests/, not a bench line)

One JSON line on rank 0 per invocation: `--config X` makes X the line's metric / value / e2e / roofline /
cpu_baseline; the default C2 line also carries compact results of C3, C4 and C5 under `other_configs` (the driver
runs the default command only) unless --no-other-configs.  A "step" = one pass of the loss path over one batch whose
logits / hidden states are resident in HBM (model forwards, generation and the optimizer are third-party code outside
the path, SURVEY.md section 8d):
  DPO step = label extraction + K1(policy) + K1(reference) + K2 + K1b (row prep + TMA-staged tile sweep) + packed all-reduce
  PPO step = rollout scoring (K3 x2, K1 x2) + rl_step (K4, K1, K5, K1b, K3 fwd/bwd, K5, pack, all-reduce)
`value` times the path with CUDA events; `e2e` drives the public trainer API with the batch (input_ids, attention_mask /
prompt + generated sequence) in pinned HOST memory copied to the device inside the timed region and the metrics read
back to the host every step.  `--impl reference` times the reference's CPU path (the oracle port of it:
/root/reference is absent on the GPU box) on the host cores, same `config` object.
`--dump-outputs DIR` writes what the timed path computed in its last step as DIR/<name>.npy (float32 / float64; tiles
too large to dump whole as a fixed, seeded sample), so that two builds can be compared output for output on the same
seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

CONFIGS = {
    'C2': dict(kind='dpo', model='Llama-3-8B (vocab 128257 after <pad> resize)', modality='text', V=128257, L=2048, pairs=32,
               modal=0, dense=True),
    'C3': dict(kind='dpo', model='LLaVA-1.5-7B', modality='image', V=32064, L=2048, pairs=32, modal=576, dense=False),
    'C5': dict(kind='dpo', model='Qwen2-Audio-7B', modality='audio', V=156032, L=4096, pairs=8, modal=750, dense=False),
    'C4': dict(kind='ppo', model='Qwen2-VL-7B', modality='image', V=152064, H=3584, prompt_len=512, max_response=512,
               prompts_per_rank=32, pad=151643),
}
SCALE_COEFF = 0.1
DPO_METRIC = 'preference-pairs/sec (DPO loss path: policy+reference log-probs, loss, grad-logits)'
PPO_METRIC = 'scored rollout-tokens/sec (PPO rollout scoring + rl_step)'


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='C2', choices=sorted(CONFIGS))
    ap.add_argument('--pairs', type=int, default=0, help='global preference pairs per step (default: the config\'s)')
    ap.add_argument('--seq-len', type=int, default=0)
    ap.add_argument('--vocab', type=int, default=0)
    ap.add_argument('--no-ppo', action='store_true')
    ap.add_argument('--no-other-configs', action='store_true')
    ap.add_argument('--no-eager-baseline', action='store_true')
    ap.add_argument('--no-ragged', action='store_true')
    ap.add_argument('--no-lm-head', action='store_true')
    ap.add_argument('--no-sft', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--cpu-seconds', type=float, default=12.0, help='target CPU time of the cpu_baseline sample')
    ap.add_argument('--variant', type=int, default=-1, help='K1 variant override (aa_logprob_set_tuning)')
    ap.add_argument('--ctas-per-sm', type=int, default=0)
    ap.add_argument('--bwd-variant', type=int, default=-1)
    ap.add_argument('--bwd-ctas-per-sm', type=int, default=0)
    ap.add_argument('--dump-outputs', metavar='DIR', default='',
                    help='after the timed steps, write the outputs of the last timed step as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs dumps the outputs of --impl ours')
    return args


def dpo_cfg(name, args):
    c = dict(CONFIGS[name])
    if name == args.config:  # size overrides apply to the selected config only
        c['pairs'] = args.pairs or c['pairs']
        c['L'] = args.seq_len or c['L']
        c['V'] = args.vocab or c['V']
    c['pad'] = c['V'] - 1
    return c


def config_object(name, c, world):
    """The `config` object of the JSON line -- built the same way by both arms (ours / reference)."""
    if c['kind'] == 'dpo':
        shape = 'dense responses (every row scored)' if c['dense'] else (
            f"{c['modal']} {c['modality']} placeholder positions in the prompt, responses ~U[L/8, (len-{c['modal']})/2]")
        return {'config_id': name,
                'workload': f"{c['model']} shapes text{'+' + c['modality'] if c['modality'] != 'text' else ''}->text DPO "
                            f"(BASELINE configs[{int(name[1]) - 1}]): V={c['V']}, seq_len={c['L']}, {c['pairs']} pairs/step global, {shape}",
                'global_batch': c['pairs'], 'seq_len': c['L'], 'vocab': c['V'], 'parallelism': f'dp{world}'}
    return {'config_id': name,
            'workload': f"{c['model']} shapes text+image->text PPO scoring + rl_step (BASELINE configs[3]): V={c['V']}, H={c['H']}, "
                        f"prompt {c['prompt_len']} (incl. vision tokens), responses ~U[64,{c['max_response']}], multimodal trainer",
            'global_batch': c['prompts_per_rank'] * world, 'prompts_per_rank': c['prompts_per_rank'],
            'seq_len': c['prompt_len'] + c['max_response'], 'vocab': c['V'], 'parallelism': f'dp{world}'}


# ---------------------------------------------------------------------------------------------------
def init_dist(n_gpus):
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    elif torch.cuda.is_available():
        torch.cuda.set_device(local)
    return rank, world, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist

        dist.barrier()


def max_over_ranks(x: float, world) -> float:
    if world == 1:
        return x
    import torch.distributed as dist

    t = torch.tensor([x], dtype=torch.float64, device='cuda')
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(x: float, world) -> float:
    if world == 1:
        return x
    import torch.distributed as dist

    t = torch.tensor([x], dtype=torch.float64, device='cuda')
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index = index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '100', '-i', str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, power, reasons = [], [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        return {'sm_mhz': statistics.median(sm), 'sm_max_mhz': max(mx), 'power_w_max': max(power),
                'samples': len(sm), 'reasons': sorted(reasons)}


def traffic_ratio(kernel):
    """dram bytes / algorithmic bytes of `kernel` from the committed ncu --set full capture (profiles/traffic.json)."""
    path = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(path):
        t = json.load(open(path)).get(kernel)
        if t:
            return t['dram_over_algorithmic'], t['source']
    return None, None


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        p = json.load(open(path))
        return float(p['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs, copy bandwidth)'
    return 6650.0, 'fallback (B200_PROFILING.md, 6.65 TB/s)'


# ---------------------------------------------------------------------------------------------------
# --dump-outputs: host copies of the last timed step's outputs, written by main() once the run is over
OUTPUTS = {}
DUMP_LIMIT_BYTES = 64 << 20


def keep_output(name, x):
    OUTPUTS[name] = x.detach().float().cpu().numpy() if torch.is_tensor(x) else np.asarray(x, dtype=np.float64)


def keep_tile_sample(name, tile, rows=16, elems=1 << 20):
    """A fixed, seeded sample of a tile too large to dump whole: `rows` whole rows (last dim) and `elems` single
    elements drawn over the whole tile."""
    gen = torch.Generator().manual_seed(0)
    flat = tile.detach().reshape(-1, tile.shape[-1])
    r = torch.randperm(flat.shape[0], generator=gen)[:rows].sort().values
    e = torch.randint(0, flat.numel(), (min(elems, flat.numel()),), generator=gen)
    keep_output(name + '_rows', flat[r.to(flat.device)])
    keep_output(name + '_elements', flat.reshape(-1)[e.to(flat.device)])


def dump_outputs(path):
    total = sum(a.nbytes for a in OUTPUTS.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f'--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit')
    os.makedirs(path, exist_ok=True)
    for name, a in OUTPUTS.items():
        np.save(os.path.join(path, f'{name}.npy'), a)


# ---------------------------------------------------------------------------------------------------
# synthetic batches (SURVEY.md section 8d): bf16 logits ~ N(0, 2.5^2), uniform labels, left padding
def synth_logits(n, L, V, device, seed, like=None, noise=0.3):
    out = torch.empty((n, L, V), dtype=torch.bfloat16, device=device)
    gen = torch.Generator(device=device).manual_seed(seed)
    for i in range(n):  # one sample at a time: bounded fp32 temporaries
        x = torch.randn((L, V), generator=gen, device=device)
        if like is None:
            out[i] = (x * 2.5).bfloat16()
        else:
            out[i] = (like[i].float() + noise * x).bfloat16()
        del x
    return out


def synth_preference_ids(n_pairs, L, V, pad, seed, ragged, modal=0):
    """(2 * n_pairs, L) ids (chosen rows first), left padded, + response_lens.  `modal` > 0: that many placeholder ids
    (V - 2) sit in the prompt of every sample (the image / audio span; they only lengthen the prompt, SURVEY.md 8d)."""
    gen = torch.Generator().manual_seed(seed)
    n = 2 * n_pairs
    ids = torch.randint(2, V - 2, (n, L), generator=gen)
    if not ragged and not modal:
        return ids, [L] * n
    lens, totals = [], []
    for i in range(n):
        total = max(int(torch.randint(L // 2, L + 1, (1,), generator=gen)), modal + 16)
        hi = max((total - modal) // 2, 4) if modal else L // 2 + 1
        lo = min(max(L // 8, 2), hi - 1)
        r = int(torch.randint(lo, hi, (1,), generator=gen))
        total = max(total, r + 1)
        ids[i, : L - min(total, L)] = pad
        if modal:
            s = L - min(total, L) + 4
            ids[i, s: s + modal] = V - 2
        lens.append(r)
        totals.append(total)
    return ids, lens


# ---------------------------------------------------------------------------------------------------
class Engine:
    """Stands in for a DeepSpeed engine whose forward has already produced the logits tile in HBM."""

    def __init__(self, out_fn, leaves=(), keep_grads=False):
        self.module = self
        self._out = out_fn
        self._leaves = leaves
        self._keep_grads = keep_grads
        self.last_grads = None
        self.optimizer = type('O', (), {'param_groups': [{'lr': 1e-6}]})()

    def __call__(self, *a, **kw):
        return self._out()

    def backward(self, loss):
        loss.backward()

    def step(self):
        if self._keep_grads:  # what an optimizer step would have consumed
            self.last_grads = [t.grad for t in self._leaves]
        for t in self._leaves:
            t.grad = None

    def train(self):
        pass

    def eval(self):
        pass


def dpo_trainer_class(modality):
    if modality == 'audio':
        from align_anything_b200.trainers.text_audio_to_text.dpo import DPOTrainer
    elif modality == 'image':
        from align_anything_b200.trainers.text_image_to_text.dpo import DPOTrainer
    else:
        from align_anything_b200.trainers.text_to_text.dpo import DPOTrainer
    return DPOTrainer


def dpo_bench(args, c, rank, world, device, extras=True, dump=False):
    """One DPO config: `value` (raw launches, CUDA events), per-kernel times, `e2e` through <modality> DPOTrainer.train_step.
    extras: also the ragged variant (dense configs) and the eager-GPU comparator.  dump: keep the outputs of the last
    timed step of the main variant for --dump-outputs."""
    from types import SimpleNamespace

    from align_anything_b200 import _lib as Lb
    from align_anything_b200 import ops
    from align_anything_b200.utils.multi_process import all_reduce_packed, fused_allreduce

    cls = dpo_trainer_class(c['modality'])
    strip, skip = cls.strip_pad_tokens, cls.skip_identical_pairs
    fused = fused_allreduce(device)
    V, L, pad = c['V'], c['L'], c['pad']
    if c['pairs'] % world:
        raise SystemExit(f"{c['pairs']} pairs/step must be divisible by the number of GPUs {world}")
    B = c['pairs'] // world  # pairs on this rank (independent units: no data-path collective)
    n = 2 * B
    policy = synth_logits(n, L, V, device, 1234 + rank)
    ref = synth_logits(n, L, V, device, 4321 + rank, like=policy)
    grad = torch.empty_like(policy)
    results = {}
    hbm_peak, peak_src = peaks()
    mode = Lb.MODE_FAITHFUL
    main = 'dense' if c['dense'] else 'modal'
    variants = [main] + (['ragged'] if (c['dense'] and extras and not args.no_ragged) else [])

    for variant in variants:
        ids_host, lens = synth_preference_ids(B, L, V, pad, 99 + rank, ragged=(variant != 'dense'),
                                              modal=c['modal'] if variant == 'modal' else 0)
        ids_host = ids_host.pin_memory()
        mask_host = (ids_host != pad).pin_memory()
        ids = ids_host.to(device)
        rows = sum(r - 1 for r in lens)
        lens_t = tuple(lens)
        labels0 = ops.strip_pad_tail(ids, lens_t, pad, strip)
        plan = ops._dpo_plan(policy, lens_t, labels0.stride(0))
        lp = torch.zeros((2,) + plan.out_shape, dtype=torch.bfloat16, device=device)
        stat = torch.empty((2, plan.n_rows), dtype=torch.float32, device=device)
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(args.steps)]
        check = {}
        last = {}

        def step(k=None, verify=False):
            labels = ops.strip_pad_tail(ids, lens_t, pad, strip)
            if k is not None:
                ev[k][0].record()
            ops._launch_fwd(policy, labels, plan, lp[0], stat[0], stat[1])
            if k is not None:
                ev[k][1].record()
            ops._launch_fwd(ref, labels, plan, lp[1], None, None)
            if k is not None:
                ev[k][2].record()
            res = last['k2'] = ops._dpo_launch(lp[0], lp[1], SCALE_COEFF, mode, ids if skip else None, True, None)  # K2: local stats
            # N > 1: the packed metrics are all-reduced over NVLink peer memory by a one-warp kernel on a side stream,
            # so its wait for the slowest rank overlaps K1b (what DPOTrainer.train_step does)
            pending = fused.all_reduce_async(res[1], max_lanes=(7,)) if fused is not None else None
            grad_seg = res[2]
            if k is not None:
                ev[k][3].record()
            ops._launch_bwd(policy, labels, plan, stat[0], stat[1], None, grad_seg, None, grad, mode)
            if k is not None:
                ev[k][4].record()
            if fused is None:
                return all_reduce_packed(res[1].clone(), max_lanes=(7,))
            out = pending.wait()
            if verify:  # the NVLink peer-memory all-reduce against NCCL on the same local vector, every rank
                want = all_reduce_packed(res[1].clone(), max_lanes=(7,))
                check['max_abs_diff'] = max(check.get('max_abs_diff', 0.0), float((out[:6] - want[:6]).abs().max()))
            return out

        for _ in range(args.warmup):
            step(verify=True)
        torch.cuda.synchronize()
        barrier(world)
        sampler = ClockSampler(torch.cuda.current_device())
        if variant == main and rank == 0:
            sampler.start()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        t0.record()
        for k in range(args.steps):
            stats_out = step(k)
        t1.record()
        torch.cuda.synchronize()
        barrier(world)
        clocks = sampler.stop() if (variant == main and rank == 0) else None
        if dump and variant == main:
            keep_output('dpo_policy_log_probs', lp[0])
            keep_output('dpo_reference_log_probs', lp[1])
            keep_output('dpo_per_pair', last['k2'][0])  # per pair: loss, better / worse sample reward, -, kept
            keep_output('dpo_stats', stats_out)
            keep_tile_sample('dpo_grad_logits', grad)
        ms = max_over_ranks(t0.elapsed_time(t1), world) / args.steps
        fwd_ms = statistics.mean((e[0].elapsed_time(e[1]) + e[1].elapsed_time(e[2])) / 2 for e in ev)
        k2_ms = statistics.mean(e[2].elapsed_time(e[3]) for e in ev)
        bwd_ms = statistics.mean(e[3].elapsed_time(e[4]) for e in ev)
        ops.check_status(device)
        rows_all = sum_over_ranks(float(rows), world)
        fwd_bytes = rows * V * 2  # algorithmic: each scored row read once (SURVEY.md 8d)
        results[variant] = dict(
            ms_per_step=ms, pairs_per_s=c['pairs'] / (ms / 1e3), rows_per_rank=rows, rows_global=rows_all,
            fwd_ms=fwd_ms, bwd_ms=bwd_ms, k2_ms=k2_ms,
            fwd_gbs=fwd_bytes / fwd_ms / 1e6, bwd_gbs=2 * rows * V * 2 / bwd_ms / 1e6,
            bwd_gbs_incl_zero_rows=(2 * rows * V * 2 + (n * L - rows - n) * V * 2) / bwd_ms / 1e6,
            step_bytes=8 * V * rows, clocks=clocks,
        )
        if fused is not None:
            d = max_over_ranks(check.get('max_abs_diff', float('nan')), world)
            if not d <= 1e-5:
                raise SystemExit(f'fused NVLink all-reduce disagrees with NCCL: max abs diff {d}')
            results['allreduce_check'] = f'NVLink peer-memory all-reduce == NCCL on {world} ranks during warm-up (max abs diff {d:.1e})'
        del lp, stat

        if variant == main:
            # ---- e2e through the public trainer API, batch in pinned host memory ----
            del grad
            torch.cuda.empty_cache()
            leaf = policy.requires_grad_(True)
            cfgs = SimpleNamespace(train_cfgs=SimpleNamespace(scale_coeff=SCALE_COEFF))
            tr = cls(cfgs, Engine(lambda: SimpleNamespace(logits=leaf), (leaf,)),
                     Engine(lambda: SimpleNamespace(logits=ref)), SimpleNamespace(pad_token_id=pad))
            ids_dev = torch.empty_like(ids)
            mask_dev = torch.empty(ids.shape, dtype=torch.bool, device=device)

            def e2e_step():
                ids_dev.copy_(ids_host, non_blocking=True)
                mask_dev.copy_(mask_host, non_blocking=True)
                batch = {'input_ids': ids_dev, 'attention_mask': mask_dev, 'meta_info': {'response_lens': lens}}
                return tr.train_step(batch)  # ends with the metrics' device->host read

            for _ in range(args.warmup):
                e2e_step()
            torch.cuda.synchronize()
            barrier(world)
            w0 = time.perf_counter()
            for _ in range(args.steps):
                metrics = e2e_step()
            torch.cuda.synchronize()
            w1 = time.perf_counter()
            barrier(world)
            e2e_ms = max_over_ranks((w1 - w0) * 1e3, world) / args.steps
            results['e2e'] = dict(ms_per_step=e2e_ms, pairs_per_s=c['pairs'] / (e2e_ms / 1e3),
                                  h2d=ids_host.numel() * 8 + mask_host.numel(), d2h=8 * 4, loss=metrics['train/loss'],
                                  api=f'{cls.__module__}.DPOTrainer.train_step')
            policy = leaf.detach()
            policy.grad = None
            leaf.grad = None
            del tr, leaf
            torch.cuda.empty_cache()
            if world == 1 and extras and not args.no_eager_baseline:
                results['eager'] = eager_gpu_dpo(policy, ref, ids, lens, B, pad, strip, skip)
            grad = torch.empty_like(policy)
    results['peak'] = (hbm_peak, peak_src)
    results['collective'] = ('none (1 GPU)' if world == 1 else 'one-shot NVLink peer-memory all-reduce (one warp, side stream, overlapped with K1b)' if fused is not None else 'one NCCL all-reduce of the packed vector')
    results['B'] = B
    results['main'] = main
    del grad, policy, ref
    torch.cuda.empty_cache()
    return results


def eager_gpu_dpo(policy, ref, ids, lens, B, pad, strip=True, skip=False, sample_pairs=2, reps=3):
    """Second comparator of SURVEY.md 8d: the reference's DPO loss path as it runs on a GPU today -- the oracle
    port (oracle/ref_port.py: the reference's ATen op sequence) executed with torch's stock CUDA kernels on a
    bounded sample of the same tiles.  A baseline leg like cpu_baseline: reported, never the product path."""
    from oracle import ref_port as O

    k = min(sample_pairs, B)
    sel = list(range(k)) + list(range(B, B + k))
    pol, rf, idk = policy[sel].clone(), ref[sel].clone(), ids[sel].clone()
    lk = [lens[i] for i in sel]
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for r in range(reps + 1):
        torch.cuda.synchronize()
        t0.record()
        out, g = O.dpo_forward_backward(pol, rf, idk, lk, pad, SCALE_COEFF, strip, skip)
        float(out['loss'].detach())
        t1.record()
        torch.cuda.synchronize()
        if r:
            times.append(t0.elapsed_time(t1))
        del out, g
    ms = statistics.median(times)
    del pol, rf
    torch.cuda.empty_cache()
    return dict(value=k / (ms / 1e3), unit='pairs/s', ms_per_pair=ms / k, kind='port (oracle/ref_port.py on ATen CUDA kernels)',
                sample_pairs=k, sample=f'{k} of {B} pairs, same tiles, median of {reps} after 1 warm-up')


def lm_head_bench(args, c, device, pairs=4, H=4096):
    """SURVEY.md 8f rank 1: lm_head x log-prob with and without the (rows, V) logits tile, on a reduced C2 batch
    (`pairs` pairs, dense): forward + backward of sum(log-probs) down to hidden states and the lm_head weight
    (`fused`: K6 forward, K6b + aa_linear_dhidden + aa_linear_dweight backward -- all tcgen05, no library GEMM), the
    no-gradient scoring path (K6 alone), and `dpo_fused_lm_head`: DPOTrainer(fused_lm_head=True).train_step end to end
    with the batch in pinned host memory."""
    from types import SimpleNamespace

    from align_anything_b200 import ops
    from align_anything_b200.trainers.text_to_text.dpo import DPOTrainer

    V, L, pad = c['V'], c['L'], c['pad']
    n = 2 * pairs
    g = torch.Generator(device=device).manual_seed(7)
    hidden = torch.randn((n, L, H), generator=g, device=device).bfloat16()
    weight = (torch.randn((V, H), generator=g, device=device) * 0.02).bfloat16()
    ids_host, lens = synth_preference_ids(pairs, L, V, pad, 5, ragged=False)
    ids = ids_host.to(device)
    out = {}

    def run(fused):
        h, w = hidden.clone().requires_grad_(True), weight.clone().requires_grad_(True)
        if fused:
            lp = ops.sequence_log_probs_from_hidden(h, w, ids, lens, pad)
        else:
            lp = ops.sequence_log_probs(torch.nn.functional.linear(h, w), ids, lens, pad)
        lp.float().sum().backward()
        return float(lp.detach().float().sum())

    for name, fused in (('materialised', False), ('fused', True)):
        run(fused)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(device)
        base = torch.cuda.memory_allocated(device)
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(3):
            val = run(fused)
        t1.record()
        torch.cuda.synchronize()
        out[name] = {'ms': t0.elapsed_time(t1) / 3, 'peak_extra_gb': (torch.cuda.max_memory_allocated(device) - base) / 1e9,
                     'sum_log_probs': val}
        torch.cuda.empty_cache()
    rows = sum(r - 1 for r in lens)
    flops = 2 * rows * H * V
    out['fused']['tflops_over_4_gemm_passes'] = 4 * flops / out['fused']['ms'] / 1e9
    out['fused']['path'] = 'K6 fwd; K6b + aa_linear_dhidden + aa_linear_dweight bwd (tcgen05, no library GEMM)' if ops._K6B else 'chunked cuBLAS + K1/K1b'

    def timed(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(reps):
            fn()
        t1.record()
        torch.cuda.synchronize()
        return t0.elapsed_time(t1) / reps

    # reference-model / rollout scoring (no gradient): K6 (one tcgen05 kernel) vs cuBLAS logits + K1
    with torch.no_grad():
        ms_k6 = timed(lambda: ops.sequence_log_probs_from_hidden(hidden, weight, ids, lens, pad))
        ms_lib = timed(lambda: ops.sequence_log_probs(torch.nn.functional.linear(hidden, weight), ids, lens, pad))
    # K6 is timed alone in a short burst here: the burst cuBLAS figure is the peak (the sustained one is reported too)
    mp = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json'))) if os.path.exists(os.path.join(ROOT, 'MEASURED_PEAKS.json')) else {}
    tpeak, tpeak_sustained = mp.get('bf16_tflops'), mp.get('bf16_tflops_sustained')
    tr_k6 = traffic_ratio('k6_fwd')
    out['no_grad_scoring'] = {
        'k6_ms': ms_k6, 'cublas_logits_plus_k1_ms': ms_lib, 'speedup': ms_lib / ms_k6,
        'roofline': {'bound': 'tensor', 'achieved': flops / ms_k6 / 1e9, 'peak': tpeak, 'unit': 'TFLOP/s',
                     'frac': (flops / ms_k6 / 1e9 / tpeak) if tpeak else None,
                     'traffic': tr_k6[0] * (rows * H * 2 + V * H * 2) if tr_k6[0] else None, 'traffic_source': tr_k6[1],
                     'kernel': 'linear_logprob_kernel<false> (K6: TMA + tcgen05.mma + LSE epilogue from TMEM)',
                     'peak_source': 'measured (MEASURED_PEAKS.json bf16_tflops: cuBLAS 8192^3 burst; kernel timed alone)',
                     'peak_sustained': tpeak_sustained,
                     'note': 'K6 time includes the row gather / scatter glue of sequence_log_probs_from_hidden'}}
    # ---- the same slice through the trainer: DPOTrainer(fused_lm_head=True).train_step, host batch -----------------
    del hidden
    torch.cuda.empty_cache()
    g2 = torch.Generator(device=device).manual_seed(8)
    hp = torch.randn((n, L, H), generator=g2, device=device).bfloat16().requires_grad_(True)
    hr = torch.randn((n, L, H), generator=g2, device=device).bfloat16()
    wp = weight.clone().requires_grad_(True)
    head = lambda w: SimpleNamespace(weight=w)

    class HiddenEngine(Engine):
        def __init__(self, h, w, leaves=()):
            super().__init__(lambda: SimpleNamespace(hidden_states=(h,)), leaves)
            self._w = w

        def get_output_embeddings(self):
            return head(self._w)

    tr = DPOTrainer(SimpleNamespace(train_cfgs=SimpleNamespace(scale_coeff=SCALE_COEFF)), HiddenEngine(hp, wp, (hp, wp)),
                    HiddenEngine(hr, weight), SimpleNamespace(pad_token_id=pad))
    tr.fused_lm_head = True
    ids_pin, mask_pin = ids_host.pin_memory(), (ids_host != pad).pin_memory()
    ids_dev, mask_dev = torch.empty_like(ids), torch.empty(ids.shape, dtype=torch.bool, device=device)

    def e2e_step():
        ids_dev.copy_(ids_pin, non_blocking=True)
        mask_dev.copy_(mask_pin, non_blocking=True)
        return tr.train_step({'input_ids': ids_dev, 'attention_mask': mask_dev, 'meta_info': {'response_lens': lens}})

    e2e_step()
    torch.cuda.synchronize()
    w0 = time.perf_counter()
    for _ in range(3):
        m = e2e_step()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - w0) * 1e3 / 3
    gemm_flops = 5 * flops  # policy: forward, recompute, d hidden, d weight; reference: forward
    out['dpo_fused_lm_head'] = {
        'metric': DPO_METRIC + ' incl. the lm_head GEMMs (no logits tile)', 'value': pairs / (e2e_ms / 1e3), 'unit': 'pairs/s',
        'ms_per_step': e2e_ms, 'e2e': {'value': pairs / (e2e_ms / 1e3), 'unit': 'pairs/s', 'h2d_bytes_per_step': ids_pin.numel() * 9,
                                       'd2h_bytes_per_step': 32, 'api': 'DPOTrainer(fused_lm_head=True).train_step'},
        'roofline': {'bound': 'tensor', 'achieved': gemm_flops / e2e_ms / 1e9, 'peak': tpeak_sustained, 'unit': 'TFLOP/s',
                     'frac': (gemm_flops / e2e_ms / 1e9 / tpeak_sustained) if tpeak_sustained else None, 'traffic': None,
                     'note': '5 GEMM passes of 2*rows*H*V flops per step (policy forward / recompute / d hidden / d weight + reference '
                             'forward), all on hand-written tcgen05 kernels; peak = sustained cuBLAS bf16 (a long step)'},
        'loss': m['train/loss']}
    out['config'] = {'pairs': pairs, 'rows': rows, 'H': H, 'V': V, 'gemm_tflop_per_pass': flops / 1e12,
                     'note': 'forward + backward to d(hidden), d(weight); the fused path runs 4 GEMM passes (forward, '
                             'recompute, d hidden, d weight), the materialised path 3'}
    return out


def sft_ce_bench(c, device, samples=8, reps=5):
    """SURVEY 8f row 4 (the loss of SupervisedTrainer.loss / ptx_step): ops.causal_lm_loss forward + backward on a
    (samples, L, V) tile of the config's shape, prompt positions ignored -- single pass (K1f, the default) against
    K1 -> mean NLL -> K1b.  An extra object: it does not enter `value`."""
    from align_anything_b200 import ops

    V, L = c['V'], c['L']
    logits = synth_logits(samples, L, V, device, 909)
    gen = torch.Generator().manual_seed(3)
    labels = torch.randint(0, V, (samples, L), generator=gen)
    prompt = torch.randint(L // 8, L // 2, (samples,), generator=gen)
    for b in range(samples):
        labels[b, : int(prompt[b])] = -100
    labels = labels.to(device)
    valid = int((labels[:, 1:] != -100).sum())
    leaf = logits.requires_grad_(True)
    out = {'config': {'samples': samples, 'seq_len': L, 'vocab': V, 'valid_rows': valid, 'tile_rows': samples * L}}
    saved = ops._FUSED_CE
    try:
        for name, flag in (('single_pass', True), ('two_pass', False)):
            ops._FUSED_CE = flag
            ts = []
            for r in range(reps + 2):
                leaf.grad = None
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                t0.record()
                loss = ops.causal_lm_loss(leaf, labels)
                loss.backward()
                t1.record()
                torch.cuda.synchronize()
                if r >= 2:
                    ts.append(t0.elapsed_time(t1))
            ms = statistics.median(ts)
            passes = 2 if flag else 3
            hbm = (valid * V * 2 * passes + (samples * L - valid) * V * 2) / 1e9
            out[name] = {'ms': ms, 'loss': float(loss.detach()), 'min_hbm_gb': hbm, 'gbs_of_min_bytes': hbm / ms * 1e3}
    finally:
        ops._FUSED_CE = saved
    ops.check_status(device)
    out['speedup'] = out['two_pass']['ms'] / out['single_pass']['ms']
    del leaf, logits
    torch.cuda.empty_cache()
    return out


def eager_gpu_ppo(actor, refl, critic_h, rm_h, w_c, w_r, seq, prompt, pad, resp, reps=2):
    """The reference's multimodal PPO scoring + rl_step arithmetic as it runs on a GPU today: the oracle port
    (per-sample Python loops, the GAE loop over time steps, ~8 tiny ATen kernels per loss) on the same tensors.
    A baseline leg: reported, never the product path."""
    from oracle import ref_port as O

    tokens = sum(resp)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for r in range(reps + 1):
        leaf = actor.clone().requires_grad_(True)
        cleaf = critic_h.clone().requires_grad_(True)
        wc = w_c.clone().requires_grad_(True)
        torch.cuda.synchronize()
        t0.record()
        out = ppo_port_step(O, actor, refl, critic_h, rm_h, w_c, w_r, seq, prompt, pad, leaf, cleaf, wc)
        float(out['actor_loss'].detach())
        t1.record()
        torch.cuda.synchronize()
        if r:
            times.append(t0.elapsed_time(t1))
        del leaf, cleaf, out
    ms = statistics.median(times)
    torch.cuda.empty_cache()
    return dict(value=tokens / (ms / 1e3), unit='tokens/s', ms_per_step=ms,
                kind='port (oracle/ref_port.py on ATen CUDA kernels)', sample=f'same batch, median of {reps} after 1 warm-up')


def ppo_port_step(O, actor, refl, critic_h, rm_h, w_c, w_r, seq, prompt, pad, leaf, cleaf, wc):
    """trainers/text_image_to_text/ppo.py actor_step bookkeeping + rollout scoring + rl_step, oracle port, any device."""
    with torch.no_grad():
        moved = O.move_padding_left(seq, pad)
        lens = O.response_lengths(prompt, seq, pad)
        rm = O.score_head(rm_h, w_r, None, 'last', False)
        cr = O.score_head(critic_h, w_c, None, 'last', False)
        roll = O.ppo_mm_rollout_scoring(actor, refl, moved, lens, rm['end_scores'].squeeze(-1), cr['scores'].squeeze(-1)[:, :-1])
    new_scores = O.score_head(cleaf, wc, None, 'last', False)['scores']
    out = O.ppo_mm_rl_step(roll, leaf, new_scores, moved)
    out['actor_loss'].backward()
    out['reward_critic_loss'].backward()
    return out


def ppo_bench(args, rank, world, device, tail=None, dump=False):
    """BASELINE configs[3].  tail: None = the trainer's default (`PPOTrainer.tail_logits`), True / False force the
    tail tile (actor / reference asked for the last max(R)+1 positions only, HF `logits_to_keep`) or the full tile.
    dump: keep the outputs of the last timed step of the resident loop for --dump-outputs."""
    from types import SimpleNamespace

    from align_anything_b200.models.reward_model import score_model_outputs
    from align_anything_b200.trainers.text_image_to_text.ppo import PPOTrainer

    c = CONFIGS['C4']
    V, H, Bp, pad = c['V'], c['H'], c['prompts_per_rank'], c['pad']
    L = c['prompt_len'] + c['max_response']
    gen = torch.Generator().manual_seed(777 + rank)
    resp = torch.randint(64, c['max_response'] + 1, (Bp,), generator=gen).tolist()
    prompt = torch.randint(2, pad, (Bp, c['prompt_len']), generator=gen)
    seq = torch.full((Bp, L), pad, dtype=torch.int64)
    seq[:, : c['prompt_len']] = prompt
    for b, r in enumerate(resp):
        seq[b, c['prompt_len'] : c['prompt_len'] + r] = torch.randint(2, pad, (r,), generator=gen)
    prompt_host, seq_host = prompt.pin_memory(), seq.pin_memory()
    tr = PPOTrainer(None, tokenizer=SimpleNamespace(pad_token_id=pad))
    if tail is not None:
        tr.tail_logits = tail
    tail = bool(tr.tail_logits)
    K = (c['max_response'] + 1) if tail else L  # what the trainer asks for: logits_to_keep = generated positions + 1
    actor = synth_logits(Bp, K, V, device, 31 + rank)
    refl = synth_logits(Bp, K, V, device, 57 + rank, like=actor)
    g2 = torch.Generator(device=device).manual_seed(5 + rank)
    critic_h = torch.randn((Bp, L, H), generator=g2, device=device).bfloat16()
    rm_h = torch.randn((Bp, L, H), generator=g2, device=device).bfloat16()
    w_c = (0.02 * torch.randn((1, H), generator=g2, device=device)).bfloat16().requires_grad_(True)
    w_r = (0.02 * torch.randn((1, H), generator=g2, device=device)).bfloat16()
    actor_leaf = actor.requires_grad_(True)
    critic_leaf = critic_h.requires_grad_(True)

    tr.actor_model = Engine(lambda: SimpleNamespace(logits=actor_leaf), (actor_leaf,), keep_grads=dump)
    tr.actor_reference_model = Engine(lambda: SimpleNamespace(logits=refl))
    tr.reward_model = Engine(lambda: score_model_outputs(rm_h, w_r, None, 'last', False))
    tr.reward_critic_model = Engine(lambda: score_model_outputs(critic_leaf, w_c, None, 'last', False), (critic_leaf, w_c),
                                    keep_grads=dump)
    prompt_dev = torch.empty((Bp, c['prompt_len']), dtype=torch.int64, device=device)
    seq_dev = torch.empty((Bp, L), dtype=torch.int64, device=device)

    last = {}

    def step(e2e: bool):
        if e2e:
            prompt_dev.copy_(prompt_host, non_blocking=True)
            seq_dev.copy_(seq_host, non_blocking=True)
        moved, attn, lens = tr.postprocess_generation(prompt_dev, seq_dev)
        inference, training = last['training'] = tr.score_rollout({'input_ids': moved, 'attention_mask': attn}, lens)
        return tr.rl_step(inference, training), lens

    prompt_dev.copy_(prompt_host)
    seq_dev.copy_(seq_host)
    out = {}
    for label, e2e in (('resident', False), ('e2e', True)):
        for _ in range(args.warmup):
            step(e2e)
        torch.cuda.synchronize()
        barrier(world)
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.perf_counter()
        t0.record()
        for _ in range(args.steps):
            metrics, lens = step(e2e)
        t1.record()
        torch.cuda.synchronize()
        w1 = time.perf_counter()
        barrier(world)
        ms_dev = max_over_ranks(t0.elapsed_time(t1), world) / args.steps
        ms_wall = max_over_ranks((w1 - w0) * 1e3, world) / args.steps
        out[label] = (ms_dev, ms_wall)
        if dump and not e2e:
            training = last['training'][1]
            for name in ('log_probs', 'ref_log_probs', 'reward', 'reward_values'):
                keep_output(f'ppo_{name}', training[name])
            for name, t in tr.last_rl_tensors.items():
                keep_output(f'ppo_{name}', t)
            for name, v in metrics.items():
                keep_output('ppo_' + name.replace('/', '_'), v)
            keep_tile_sample('ppo_grad_actor_logits', tr.actor_model.last_grads[0])
            keep_tile_sample('ppo_grad_critic_hidden', tr.reward_critic_model.last_grads[0])
            keep_output('ppo_grad_critic_head', tr.reward_critic_model.last_grads[1])
    eager = None
    if world == 1 and not tail and not getattr(args, 'no_eager_baseline', False):
        eager = eager_gpu_ppo(actor_leaf.detach(), refl, critic_h.detach(), rm_h, w_c.detach(), w_r, seq_dev, prompt_dev, pad, resp)
    tokens_rank = sum(resp)
    assert list(lens) == resp
    tokens = sum_over_ranks(float(tokens_rank), world)
    hbm_peak, _ = peaks()
    ms = out['resident'][0]
    bytes_token = 10 * V + 10 * H + 40
    tr_ppo = traffic_ratio('ppo_step')
    cfg = config_object('C4', c, world)
    cfg.update({'logits_rows_per_sample': K, 'scored_tokens_per_step': int(tokens), 'tail_logits': tail})
    res = dict(
        metric=PPO_METRIC, value=tokens / (ms / 1e3), unit='tokens/s', ms_per_step=ms, n_gpus=world, scaling='weak',
        e2e={'value': tokens / (out['e2e'][1] / 1e3), 'unit': 'tokens/s',
             'h2d_bytes_per_step': (prompt_host.numel() + seq_host.numel()) * 8, 'd2h_bytes_per_step': 12 * 4,
             'api': 'PPOTrainer.postprocess_generation -> score_rollout -> rl_step (text_image_to_text mirror)'},
        config=cfg,
        roofline={'bound': 'hbm', 'achieved': tokens / world * bytes_token / (ms / 1e3) / 1e9, 'peak': hbm_peak, 'unit': 'GB/s',
                  'frac': tokens / world * bytes_token / (ms / 1e3) / 1e9 / hbm_peak,
                  'traffic': tr_ppo[0] * tokens / world * bytes_token if tr_ppo[0] else None, 'traffic_source': tr_ppo[1],
                  'note': 'algorithmic 10*V + 10*H + 40 bytes per scored token (SURVEY.md 8d); the zero rows of the '
                          'gradient tile are written but not counted; the actor node (K1f) reads the scored rows once '
                          'for log-prob AND gradient, so the measured DRAM traffic can fall below 10*V per token'},
        actor_loss=metrics['train/actor_loss'],
    )
    if eager is not None:
        res['gpu_eager_baseline'] = eager
    return res


# ---------------------------------------------------------------------------------------------------
def _pick_threads(run_probe, threads):
    """The reference's per-sample Python loops do not scale to every core of a big host: probe a few thread counts and
    keep the fastest (all cores is always one of the candidates)."""
    best = None
    for th in sorted({threads, min(threads, 64), min(threads, 32), min(threads, 16)}, reverse=True):
        torch.set_num_threads(th)
        run_probe(True)  # warm-up
        t = run_probe(False)
        if best is None or t < best[1]:
            best = (th, t)
    torch.set_num_threads(best[0])
    return best


def cpu_dpo_pairs_per_s(c, target_s, threads):
    """The reference's CPU trainer path for one DPO unit (oracle port of DPOTrainer.loss + backward to the policy
    logits, text / image / audio variant) on a bounded sample: 1 pair of a shortened dense sequence, converted to
    pairs/s of the config by scored rows (the work is linear in them)."""
    from oracle import ref_port as O

    V, L = c['V'], c['L']
    strip, skip = c['modality'] != 'audio', c['modality'] == 'audio'
    gen = torch.Generator().manual_seed(0)

    def run(Lc):
        ids = torch.randint(2, V - 1, (2, Lc), generator=gen)
        pol = (torch.randn(2, Lc, V, generator=gen) * 2.5).bfloat16()
        ref = (pol.float() + 0.3 * torch.randn(2, Lc, V, generator=gen)).bfloat16()
        t = time.perf_counter()
        O.dpo_forward_backward(pol, ref, ids, [Lc, Lc], V - 1, SCALE_COEFF, strip, skip)
        return time.perf_counter() - t

    probe_L = 64
    th, t_probe = _pick_threads(lambda warm: run(8 if warm else probe_L), threads)
    per_row = t_probe / (2 * (probe_L - 1))
    cpu_dpo_pairs_per_s.threads_used = th
    ids_all, lens_all = synth_preference_ids(c['pairs'], L, V, c['pad'], 99, ragged=not c['dense'], modal=c['modal'])
    rows_per_pair = sum(r - 1 for r in lens_all) / c['pairs']
    if per_row * 2 * (L - 1) <= 4 * target_s:
        # pair 0 of the very batch the GPU arm runs (rank 0), at the real sequence length: the reference's per-sample slice
        # backward pads each slice back into a full (L, V) tile, so its cost is not a function of the scored rows alone
        B = c['pairs']
        ids = ids_all[[0, B]]
        lens = [lens_all[0], lens_all[B]]
        pol = (torch.randn(2, L, V, generator=gen) * 2.5).bfloat16()
        ref = (pol.float() + 0.3 * torch.randn(2, L, V, generator=gen)).bfloat16()
        t0 = time.perf_counter()
        O.dpo_forward_backward(pol, ref, ids, lens, c['pad'], SCALE_COEFF, strip, skip)
        t = time.perf_counter() - t0
        scale = (sum(lens) - 2) / rows_per_pair  # this pair's scored rows vs the batch mean
        return scale / t, (f'1 pair of the batch at full size (seq_len {L}, V={V}, responses {lens[0]} + {lens[1]} tokens), {t:.2f} s on '
                           f'{th} of {threads} host threads (fastest of the probed counts); x{scale:.2f} for the batch-mean scored rows')
    Lc = int(min(L, max(probe_L, target_s / per_row / 2 + 1)))
    t = run(Lc)
    pairs_per_s = (2 * (Lc - 1) / t) / rows_per_pair
    return pairs_per_s, (f'1 pair, dense, seq_len {Lc} (V={V}), {t:.2f} s on {th} of {threads} host threads (fastest of the probed '
                         f'counts); converted by scored rows ({2 * (Lc - 1)} in the sample, {rows_per_pair:.0f} per pair of the config)')


def cpu_ppo_tokens_per_s(target_s, threads):
    """The reference's CPU path for the PPO unit (oracle port of the multimodal actor_step bookkeeping + rollout scoring
    + rl_step incl. both backwards) on a bounded sample: 1 prompt, full V and H, prompt : response lengths in the
    config's mean ratio (the per-sample slice backward pads every gradient back to the whole (L, V) tile)."""
    from oracle import ref_port as O

    c = CONFIGS['C4']
    V, H, pad = c['V'], c['H'], c['pad']
    gen = torch.Generator().manual_seed(0)

    def run(R):
        P = max(int(R * c['prompt_len'] / ((64 + c['max_response']) / 2)), 2)
        Lc = P + R
        prompt = torch.randint(2, pad, (1, P), generator=gen)
        seq = torch.cat([prompt, torch.randint(2, pad, (1, R), generator=gen)], dim=1)
        actor = (torch.randn(1, Lc, V, generator=gen) * 2.5).bfloat16()
        refl = (actor.float() + 0.3 * torch.randn(1, Lc, V, generator=gen)).bfloat16()
        critic_h, rm_h = torch.randn(1, Lc, H, generator=gen).bfloat16(), torch.randn(1, Lc, H, generator=gen).bfloat16()
        w_c, w_r = (0.02 * torch.randn(1, H, generator=gen)).bfloat16(), (0.02 * torch.randn(1, H, generator=gen)).bfloat16()
        leaf, cleaf, wc = actor.clone().requires_grad_(True), critic_h.clone().requires_grad_(True), w_c.clone().requires_grad_(True)
        t = time.perf_counter()
        ppo_port_step(O, actor, refl, critic_h, rm_h, w_c, w_r, seq, prompt, pad, leaf, cleaf, wc)
        return time.perf_counter() - t, P

    th, t_probe = _pick_threads(lambda warm: run(4 if warm else 16)[0], threads)
    R = int(min(c['max_response'], max(16, target_s / (t_probe / 16))))
    t, P = run(R)
    cpu_ppo_tokens_per_s.threads_used = th
    return R / t, (f'1 prompt, prompt {P} + response {R} tokens (V={V}, H={H}), {t:.2f} s on {th} of {threads} host threads '
                   f'(fastest of the probed counts)')


def reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path.  /root/reference is not on the GPU box and
    the reference is pure Python on torch, so this runs the oracle port of it (oracle/ref_port.py, pinned bit-exactly on
    the reference's outputs) on the host cores.  Each step = one bounded sample; same `config` object as our arm."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    world = int(os.environ.get('WORLD_SIZE', '1'))
    threads = os.cpu_count() or 1
    per_step_s = max(1.0, min(6.0, 90.0 / max(args.steps + args.warmup, 1)))
    name = args.config
    c = dpo_cfg(name, args) if CONFIGS[name]['kind'] == 'dpo' else CONFIGS[name]
    vals, walls, sample = [], [], ''
    for i in range(args.warmup + args.steps):
        w0 = time.perf_counter()
        if c['kind'] == 'dpo':
            v, sample = cpu_dpo_pairs_per_s(c, per_step_s, threads)
            used = cpu_dpo_pairs_per_s.threads_used
        else:
            v, sample = cpu_ppo_tokens_per_s(per_step_s, threads)
            used = cpu_ppo_tokens_per_s.threads_used
        if i >= args.warmup:
            vals.append(v)
            walls.append(time.perf_counter() - w0)
    value = statistics.mean(vals)
    unit = 'pairs/s' if c['kind'] == 'dpo' else 'tokens/s'
    # a reference-arm "step" is ONE bounded sample (thread probing + one pair / prompt), not a whole batch: ms_per_step
    # is its wall time, so steps x ms_per_step is the time this arm really ran; a whole batch would take
    # `full_batch_ms` at the measured rate
    step_ms = 1e3 * statistics.mean(walls)
    line = {
        'impl': 'reference', 'metric': DPO_METRIC if c['kind'] == 'dpo' else PPO_METRIC,
        'value': value, 'unit': unit, 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': step_ms, 'full_batch_ms': (1e3 * c['pairs'] / value) if c['kind'] == 'dpo' else None,
        'higher_is_better': True,
        'scaling': 'strong' if c['kind'] == 'dpo' else 'weak', 'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
        'config': config_object(name, c, world),
        'cpu_baseline': {'value': value, 'unit': unit, 'cores': used, 'kind': 'port', 'sample': sample,
                         'sample_pairs': 1 if c['kind'] == 'dpo' else None},
        'e2e': {'value': value, 'unit': unit, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    if name == 'C2' and not args.no_ppo:  # the default command also reports the PPO unit of the reference's CPU path
        v, s = cpu_ppo_tokens_per_s(per_step_s, threads)
        line['ppo'] = {'metric': PPO_METRIC, 'value': v, 'unit': 'tokens/s',
                       'cpu_baseline': {'value': v, 'unit': 'tokens/s', 'cores': cpu_ppo_tokens_per_s.threads_used, 'kind': 'port', 'sample': s}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
def dpo_line(args, name, c, dpo, world, cpu):
    d = dpo[dpo['main']]
    hbm_peak, peak_src = dpo['peak']
    V = c['V']
    t_f, t_b = traffic_ratio('k1_fwd'), traffic_ratio('k1b_bwd')
    line = {
        'metric': DPO_METRIC, 'value': d['pairs_per_s'], 'unit': 'pairs/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': d['ms_per_step'], 'higher_is_better': True, 'scaling': 'strong',
        'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
        'config': config_object(name, c, world),
        'details': {'pairs_per_rank': dpo['B'], 'scored_rows_per_rank': d['rows_per_rank'],
                    'l2': 'inputs (2 x %.1f GB logits tiles per rank) are far larger than the 126 MB L2; no flush needed'
                          % (2 * dpo['B'] * c['L'] * V * 2 / 1e9),
                    'rounding': 'faithful (reference bf16 rounding points)', 'collective': dpo['collective'],
                    'allreduce_check': dpo.get('allreduce_check')},
        'gpu_launches': args.steps * 6,  # strip_pad_tail, K1 x2, K2, K1b row-prep, K1b
        'e2e': {'value': dpo['e2e']['pairs_per_s'], 'unit': 'pairs/s', 'h2d_bytes_per_step': dpo['e2e']['h2d'],
                'd2h_bytes_per_step': dpo['e2e']['d2h'], 'ms_per_step': dpo['e2e']['ms_per_step'],
                'api': dpo['e2e']['api'] + ' (input_ids + attention_mask from pinned host memory, metrics read back; logits '
                       'are produced on-device by the model forward in the reference and are resident here)'},
        'roofline': {'bound': 'hbm', 'achieved': d['fwd_gbs'], 'peak': hbm_peak, 'unit': 'GB/s', 'frac': d['fwd_gbs'] / hbm_peak,
                     'traffic': (t_f[0] * d['rows_per_rank'] * V * 2) if t_f[0] else None, 'traffic_source': t_f[1],
                     'kernel': 'logprob_fwd_kernel (K1)', 'peak_source': peak_src,
                     'bytes_per_launch': d['rows_per_rank'] * V * 2, 'launch_ms': d['fwd_ms'], 'peak_nominal': 8000.0,
                     'frac_of_nominal': d['fwd_gbs'] / 8000.0},
        'roofline_bwd': {'bound': 'hbm', 'achieved': d['bwd_gbs'], 'peak': hbm_peak, 'unit': 'GB/s',
                         'frac': d['bwd_gbs'] / hbm_peak, 'kernel': 'logprob_bwd_tma_kernel (K1b)', 'launch_ms': d['bwd_ms'],
                         'bytes_per_launch': 2 * d['rows_per_rank'] * V * 2,
                         'achieved_incl_zero_rows': d['bwd_gbs_incl_zero_rows'],
                         'traffic': (t_b[0] * 2 * d['rows_per_rank'] * V * 2) if t_b[0] else None},
        'step_roofline_frac': d['step_bytes'] / (d['ms_per_step'] / 1e3) / 1e9 / hbm_peak,
        'kernel_ms': {'k1_fwd': d['fwd_ms'], 'k2_dpo': d['k2_ms'], 'k1b_bwd': d['bwd_ms']},
        'clocks': d['clocks'],
        'cpu_baseline': cpu,
    }
    if 'ragged' in dpo:
        r = dpo['ragged']
        line['ragged'] = {'value': r['pairs_per_s'], 'unit': 'pairs/s', 'ms_per_step': r['ms_per_step'],
                          'rows_per_rank': r['rows_per_rank'], 'fwd_gbs': r['fwd_gbs'], 'bwd_gbs': r['bwd_gbs'],
                          'bwd_gbs_incl_zero_rows': r['bwd_gbs_incl_zero_rows'],
                          'note': 'R_i ~ U[L/8, L/2]; the gradient tile is still (2B, L, V): unscored rows are zero-filled'}
    if 'eager' in dpo:
        line['gpu_eager_baseline'] = dpo['eager']
    return line


def compact(line):
    keep = ('metric', 'value', 'unit', 'ms_per_step', 'n_gpus', 'scaling', 'config', 'e2e', 'roofline', 'roofline_bwd',
            'step_roofline_frac', 'kernel_ms', 'cpu_baseline', 'gpu_eager_baseline', 'error')
    return {k: line[k] for k in keep if k in line}


def main():
    args = parse()
    if args.impl == 'reference':
        reference_arm(args)
        return
    if not torch.cuda.is_available():
        raise SystemExit('bench.py --impl ours needs a B200: the product path has no CPU fallback')
    rank, world, local = init_dist(args.gpus)
    device = torch.device('cuda', local)
    from align_anything_b200 import _lib as Lb

    if args.variant >= 0 or args.ctas_per_sm > 0:
        Lb.check(Lb.lib().aa_logprob_set_tuning(max(args.variant, 0), args.ctas_per_sm))
        Lb.check(Lb.lib().aa_logprob_set_tuning_bwd(0, 0))  # keep the backward on its own defaults
    if args.bwd_variant >= 0:
        Lb.check(Lb.lib().aa_logprob_set_tuning_bwd(args.bwd_variant, args.bwd_ctas_per_sm))
    threads = os.cpu_count() or 1
    solo = rank == 0 and world == 1

    def cpu_dpo(c, seconds):
        if not solo or args.no_cpu_baseline:
            return None
        v, sample = cpu_dpo_pairs_per_s(c, seconds, threads)
        return {'value': v, 'unit': 'pairs/s', 'cores': cpu_dpo_pairs_per_s.threads_used, 'kind': 'port', 'sample': sample,
                'sample_pairs': 1}

    def cpu_ppo(seconds):
        if not solo or args.no_cpu_baseline:
            return None
        v, sample = cpu_ppo_tokens_per_s(seconds, threads)
        return {'value': v, 'unit': 'tokens/s', 'cores': cpu_ppo_tokens_per_s.threads_used, 'kind': 'port', 'sample': sample}

    dump = bool(args.dump_outputs) and rank == 0

    def run_ppo(full):
        ppo = ppo_bench(args, rank, world, device, dump=dump)
        torch.cuda.empty_cache()
        if full:
            other = ppo_bench(args, rank, world, device, tail=not ppo['config']['tail_logits'])
            key = 'tail_logits_variant' if other['config']['tail_logits'] else 'full_tile_variant'
            ppo[key] = {k: other[k] for k in ('value', 'unit', 'ms_per_step', 'config', 'roofline') if k in other}
            if 'gpu_eager_baseline' in other:
                ppo['gpu_eager_baseline'] = other['gpu_eager_baseline']
            ppo[key]['note'] = ('PPOTrainer.tail_logits=True: the models return logits for the last max(R)+1 positions only (HF '
                                'logits_to_keep); False: whole (B, L, V) tiles, prompt rows of the gradient tile zero-filled')
            torch.cuda.empty_cache()
        ppo['cpu_baseline'] = cpu_ppo(min(args.cpu_seconds, 8.0))
        ppo.update({'steps': args.steps, 'warmup': args.warmup, 'higher_is_better': True, 'dtype': 'bf16', 'data': 'synthetic',
                    'vs_baseline': None})
        return ppo

    name = args.config
    if CONFIGS[name]['kind'] == 'ppo':
        line = run_ppo(full=True)
    else:
        c = dpo_cfg(name, args)
        dpo = dpo_bench(args, c, rank, world, device, dump=dump)
        line = None
        ppo = lm_head = sft = None
        others = {}
        if name == 'C2':
            if not args.no_ppo:
                try:
                    ppo = run_ppo(full=True)
                except Exception as e:  # the DPO headline must still be reported
                    ppo = {'error': repr(e)}
                torch.cuda.empty_cache()
            if not args.no_other_configs:
                for other in ('C3', 'C5'):
                    try:
                        oc = dpo_cfg(other, args)
                        od = dpo_bench(args, oc, rank, world, device, extras=False)
                        others[other] = compact(dpo_line(args, other, oc, od, world, cpu_dpo(oc, min(args.cpu_seconds, 6.0))))
                    except Exception as e:
                        others[other] = {'error': repr(e)}
                    torch.cuda.empty_cache()
                if ppo is not None:
                    others['C4'] = compact(ppo)
            if solo and not args.no_lm_head:
                try:
                    torch.cuda.empty_cache()
                    lm_head = lm_head_bench(args, c, device)
                except Exception as e:
                    lm_head = {'error': repr(e)}
            if solo and not args.no_sft:
                try:
                    torch.cuda.empty_cache()
                    sft = sft_ce_bench(c, device)
                except Exception as e:
                    sft = {'error': repr(e)}
        line = dpo_line(args, name, c, dpo, world, cpu_dpo(c, args.cpu_seconds))
        if sft is not None:
            line['sft_cross_entropy'] = sft
        if ppo is not None:
            line['ppo'] = ppo
        if others:
            line['other_configs'] = others
        if lm_head is not None:
            line['lm_head_fused'] = lm_head
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()
    if dump:
        dump_outputs(args.dump_outputs)
    if rank == 0:
        print(json.dumps(line), flush=True)


if __name__ == '__main__':
    main()
