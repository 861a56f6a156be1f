"""Functional layer over libaa_b200.so: torch tensors in, torch tensors out, autograd wired.

Every function cites the reference function whose arithmetic it replaces (paths relative to
the reference's align_anything/).  PyTorch is used for device memory, streams and autograd
plumbing only; all arithmetic on the path runs in the hand-written sm_100a kernels.

`mode`:
  'faithful' (default for 16-bit tensors) -- fp32 arithmetic, rounded to the tensor dtype at the
             points where the reference's eager ops round (results carry the reference's dtypes);
  'f32'      -- fp32 outputs, no intermediate rounding.
"""
from __future__ import annotations

import functools
import os
from typing import Sequence

import torch

from . import _lib as L

__all__ = [
    'gather_log_probabilities', 'masked_mean', 'sequence_log_probs', 'RowPlan', 'DeviceLens', 'DevicePlan', 'as_device_lens', 'rollout_layout', 'response_tail_log_probs', 'response_tail_log_probs_pair', 'dpo_loss_from_log_probs',
    'dpo_fused_loss', 'score_head', 'score_end', 'kl_rewards_and_gae', 'gae_from_rewards', 'actor_loss', 'critic_loss',
    'move_padding_left', 'count_nonpad', 'strip_pad_tail', 'ppo_pack_metrics', 'check_status', 'raise_for_status', 'status_lane', 'causal_lm_loss', 'rm_pair_loss', 'group_advantages', 'grpo_loss', 'tail_token_log_probs', 'pair_slices', 'slice_sums', 'tail_rows', 'linear_token_log_probs',
    'sequence_log_probs_from_hidden', 'fused_linear_token_log_probs', 'tail_log_probs_from_hidden', 'tail_actor_loss', 'tail_critic_loss', 'lm_head_weight',
    'CERows', 'ce_rows', 'causal_lm_loss_from_hidden', 'causal_lm_loss_from_hidden_scaled',
]

_REROUTE_TO_BASE = os.environ.get('AA_B200_REROUTE_BASE', '1') != '0'
_K6B = os.environ.get('AA_B200_K6B', '1') != '0'  # 0: lm_head path with gradient through chunked cuBLAS + K1 / K1b instead of the tcgen05 kernels
_K6 = os.environ.get('AA_B200_K6', '1') != '0'  # 0: no-grad lm_head scoring through chunked cuBLAS + K1 instead of K6
_ZERO_SPANS = os.environ.get('AA_B200_ZERO_SPANS', '1') != '0'  # 0: K1b zero-fills every unscored tile row itself
_FUSED_ACTOR = os.environ.get('AA_B200_FUSED_ACTOR', '1') != '0'  # 0: the PPO actor node runs K1 -> K5 -> K1b instead of the single-pass K1f
# fp16 logits keep the two-pass path by default: under fp16 training the incoming scalar is the loss scale (2^16 ...), and the
# two-pass backward folds it into the per-row gradient BEFORE the tile is rounded to fp16; a tile born unscaled would lose its
# small entries to fp16 underflow -- exactly what loss scaling is there to prevent.  bf16 / fp32 have the exponent range.
_FUSED_F16 = os.environ.get('AA_B200_FUSED_F16', '0') == '1'
# K1f keeps ONE row per SM in flight (that is what makes its second pass an L2 hit), so its per-row costs -- two block
# reductions, the boundary thread, ring fill / drain -- weigh more the shorter the row is.  Measured on 32 x 513 x V bf16
# actor tiles (profiles/r02_k1f_experiments.txt, call V): V = 32064: 0.83x of the two-pass path, 65536: 0.93x,
# 128256: 1.15x, 152064: 1.25x.  Rows below this many bytes keep K1 -> loss kernel -> K1b.
_FUSED_MIN_ROW_BYTES = int(os.environ.get('AA_B200_FUSED_MIN_ROW_BYTES', str(192 * 1024)))
_FUSED_GRPO = os.environ.get('AA_B200_FUSED_GRPO', '1') != '0'  # 0: the GRPO loss runs K1 -> loss kernel -> K1b instead of the single-pass K1f
_FUSED_CE = os.environ.get('AA_B200_FUSED_CE', '1') != '0'  # 0: causal_lm_loss runs K1 -> mean NLL -> K1b instead of the single-pass K1f


def _mode_code(mode: str | None, dtype: torch.dtype) -> int:
    if mode is None:
        mode = 'faithful'
    if mode == 'faithful':
        return L.MODE_FAITHFUL
    if mode == 'f32':
        return L.MODE_F32
    raise ValueError(f"mode must be 'faithful' or 'f32', got {mode!r}")


# ---- per-device scratch (status word, last-block counters) ---------------------------------------
_scratch: dict = {}


def _device_scratch(device: torch.device):
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    s = _scratch.get(key)
    if s is None:
        s = {
            'status': torch.zeros(1, dtype=torch.int32, device=device),
            'counter': torch.zeros(8, dtype=torch.int32, device=device),
        }
        _scratch[key] = s
    return s


def raise_for_status(code, device=None, reset: bool = True) -> int:
    """`code` is the status word as it came back with a step's metrics (lane 7 of the DPO stats, lane 10 of the PPO
    stats; MAX-reduced across ranks, so every rank raises together).  Raises the error the reference would have raised
    eagerly; no host sync of its own.  trainers/*: called after the ONE `.tolist()` of the step."""
    v = int(code)
    if v and reset:
        device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        _device_scratch(device)['status'].zero_()
    return _raise_status_bits(v)


def status_lane(device) -> torch.Tensor:
    """The device status word as an fp32 (1,) tensor, to be concatenated to a step's metric vector (MAX lane) so that
    the step's ONE host read also reports what the reference would have raised on; see raise_for_status."""
    return _device_scratch(torch.device(device))['status'].float()


def check_status(device=None, reset: bool = True) -> int:
    """Read the device status word (ONE host sync).  Raises the error the reference would have
    raised eagerly: out-of-range labels (torch.gather), short sequences, empty mask rows."""
    device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
    st = _device_scratch(device)['status']
    v = int(st.item())
    if reset and v:
        st.zero_()
    return _raise_status_bits(v)


def _raise_status_bits(v: int) -> int:
    if v & L.STATUS_LABEL_OOB:
        raise IndexError('align_anything_b200: a label is outside [0, vocab) (torch.gather would raise)')
    if v & L.STATUS_SHORT_SEQUENCE:
        raise ValueError('align_anything_b200: a sequence has fewer non-pad tokens than its response_len')
    if v & L.STATUS_EMPTY_MASK:
        raise IndexError('align_anything_b200: a mask row has no True element (m.nonzero()[-1] would raise)')
    if v & L.STATUS_DIVERGE_RANGE:
        raise AssertionError('diverge index is out of range!')  # trainers/text_to_text/simpo.py:72-73
    return v


def _single_pass_ok(logits: torch.Tensor) -> bool:
    """Whether the single-pass nodes (K1f) take this tile: not fp16 (the tile is written for an upstream gradient of 1 and
    scaled afterwards, see _FUSED_F16) and rows long enough for K1f to win (see _FUSED_MIN_ROW_BYTES)."""
    if logits.dtype == torch.float16 and not _FUSED_F16:
        return False
    return logits.size(-1) * logits.element_size() >= _FUSED_MIN_ROW_BYTES


# ---- row plans -----------------------------------------------------------------------------------
class RowPlan:
    """Which logits rows are scored against which labels, and where the results go.

    Segment s = n[s] consecutive rows starting at element offset logit_off[s] (stride row_stride)
    of the logits tensor, labels starting at label_off[s], outputs at out_off[s] of the flat
    output buffer; tile_row[s] is the row index of the segment's first row in the gradient tile
    (the logits tensor viewed as (n_tile_rows, V))."""

    __slots__ = ('n_seg', 'n_rows', 'dev', 'out_shape', 'n_tile_rows', 'zero_spans', 'n_zero_spans', 'extra_zero_rows',
                 'n_extra')
    exact = True        # n_rows is the exact number of scored rows
    host_layout = True  # the complement of the segments is known on the host (memset spans / listed zero rows)

    # zero spans of at least this many rows go to the copy engine (cudaMemsetAsync, aa_zero_rows); shorter ones
    # are listed for the kernel (a memset launch costs ~2-3 us, a 256 KB row 40 ns of HBM time)
    MEMSET_MIN_ROWS = 16

    def __init__(self, logit_off, label_off, out_off, counts, tile_row, out_shape, n_tile_rows, device):
        n_seg = len(counts)
        cum = [0] * (n_seg + 1)
        for i, c in enumerate(counts):
            if c < 0:
                raise ValueError('negative row count in RowPlan')
            cum[i + 1] = cum[i] + c
        self.n_seg = n_seg
        self.n_rows = cum[-1]
        table = torch.tensor(
            [list(logit_off) + [0], list(label_off) + [0], list(out_off) + [0], cum, list(tile_row) + [0]],
            dtype=torch.int64,
        )
        self.dev = table.to(device, non_blocking=True)  # (5, n_seg+1)
        self.out_shape = tuple(out_shape)
        self.n_tile_rows = int(n_tile_rows)
        # complement of the segments inside the gradient tile, known on the host: (first_row, n_rows) spans
        self.zero_spans, self.n_zero_spans, self.extra_zero_rows, self.n_extra = None, 0, None, 0
        if self.n_tile_rows > 0:
            import ctypes

            big, small, at = [], [], 0
            for first, n in sorted((int(t), int(c)) for t, c in zip(tile_row, counts) if c > 0):
                if first < at:
                    raise ValueError('RowPlan segments overlap in the gradient tile')
                if first > at:
                    (big if first - at >= self.MEMSET_MIN_ROWS else small).append((at, first - at))
                at = first + n
            if at > self.n_tile_rows:
                raise ValueError('RowPlan segments exceed the gradient tile')
            if at < self.n_tile_rows:
                (big if self.n_tile_rows - at >= self.MEMSET_MIN_ROWS else small).append((at, self.n_tile_rows - at))
            flat = [v for span in big for v in span]
            self.zero_spans = (ctypes.c_int64 * max(len(flat), 1))(*flat)
            self.n_zero_spans = len(big)
            rows = [r for first, n in small for r in range(first, first + n)]
            self.n_extra = len(rows)
            if rows:
                self.extra_zero_rows = torch.tensor(rows, dtype=torch.int64).to(device, non_blocking=True)

    def ptrs(self):
        base = self.dev.data_ptr()
        step = self.dev.stride(0) * 8
        return base, base + step, base + 2 * step, base + 3 * step, base + 4 * step


class DeviceLens:
    """Per-sample response lengths that live on the DEVICE (int32 (B,)) plus a host-known upper bound -- what
    PPOTrainer.postprocess_generation returns instead of the reference's Python list
    (trainers/text_image_to_text/ppo.py:190-203).  Everything on the path takes the device tensor; the list protocol
    (`len`, iteration, indexing, `==`, `tolist`) is kept for reference code that reads `training_batch['response_lens']`
    and costs ONE host sync on first use."""

    __slots__ = ('dev', 'bound', '_host', '_plans')

    def __init__(self, dev: torch.Tensor, bound: int, host=None):
        self.dev = dev
        self.bound = int(bound)
        self._host = list(host) if host is not None else None
        self._plans = {}  # row plans built from these lengths (ops.device_tail_plan): one build per distinct tile layout

    def tolist(self):
        if self._host is None:
            self._host = self.dev.tolist()
        return self._host

    def __len__(self):
        return self.dev.numel()

    def __iter__(self):
        return iter(self.tolist())

    def __getitem__(self, i):
        return self.tolist()[i]

    def __eq__(self, other):
        return self.tolist() == list(other)

    def __repr__(self):
        return f'DeviceLens(B={len(self)}, bound={self.bound}, host={self._host})'


def device_tail_plan(lens: 'DeviceLens', *key) -> 'DevicePlan':
    """DevicePlan(lens, *key), built once per DeviceLens object and tile layout: the rollout (actor, reference) and the
    rl_step (actor) of one PPO step address tiles of the same shape, so one aa_tail_plan_build launch serves all three."""
    plan = lens._plans.get(key)
    if plan is None:
        plan = lens._plans[key] = DevicePlan(lens, *key)
    return plan


def as_device_lens(lens, device) -> DeviceLens:
    """A host list of lengths -> DeviceLens with the exact bound (one cached H2D copy, no sync)."""
    if isinstance(lens, DeviceLens):
        return lens
    host = tuple(int(r) for r in lens)
    return DeviceLens(_lens_tensor(host, str(device)), max(max(host), 1) if host else 1, host)


class DevicePlan:
    """RowPlan whose table is built ON THE DEVICE from DeviceLens (aa_tail_plan_build): n_rows is an upper bound (the
    kernels read the exact count from the table), the backward runs in tile mode (the prep kernel orders the work list:
    scored rows first, zero rows after), nothing about the row layout is known on the host."""

    __slots__ = ('n_seg', 'n_rows', 'dev', 'out_shape', 'n_tile_rows')
    exact = False        # out buffers must be zero-initialised: rows beyond a sample's length are padding
    host_layout = False  # no memset spans: K1b zero-fills every unscored tile row itself

    def __init__(self, lens: DeviceLens, seq: int, sample_stride: int, row_stride: int, label_row_stride: int,
                 label_tail_len: int, label_shift: int, row_shift: int, width: int, copies: int = 1,
                 copy_logit_delta: int = 0):
        B = len(lens)
        dev = lens.dev.device
        S = B * copies
        self.n_seg, self.n_rows, self.n_tile_rows = S, S * width, S * seq
        self.out_shape = (B, width) if copies == 1 else (copies, B, width)
        self.dev = torch.empty((5, S + 1), dtype=torch.int64, device=dev)
        L.check(L.lib().aa_tail_plan_build(lens.dev.data_ptr(), B, int(seq), int(sample_stride), int(row_stride),
                                           int(label_row_stride), int(label_tail_len), int(label_shift), int(row_shift),
                                           int(width), int(copies), int(copy_logit_delta), B * int(width),
                                           self.dev.data_ptr(), _device_scratch(dev)['status'].data_ptr(), L.stream_ptr(dev)))

    def ptrs(self):
        base = self.dev.data_ptr()
        step = self.dev.stride(0) * 8
        return base, base + step, base + 2 * step, base + 3 * step, base + 4 * step


@functools.lru_cache(maxsize=256)
def _dense_plan(B, rows, sb, sl, lab_sb, tile_row0, tile_sb, n_tile_rows, device_str):
    """Plan for a (B, rows, V) view: every row of every sample is scored."""
    device = torch.device(device_str)
    if B > 0 and sb == rows * sl and lab_sb == rows and tile_sb == rows:
        # rows are uniformly strided across samples: a single segment
        return RowPlan([0], [0], [0], [B * rows], [tile_row0], (B, rows), n_tile_rows, device)
    return RowPlan(
        [b * sb for b in range(B)], [b * lab_sb for b in range(B)], [b * rows for b in range(B)],
        [rows] * B, [tile_row0 + b * tile_sb for b in range(B)], (B, rows), n_tile_rows, device,
    )


@functools.lru_cache(maxsize=256)
def _tail_plan(lens: tuple, L_seq: int, sb: int, sl: int, lab_stride: int, lab_shift: int, row_shift: int,
               width: int | None, device_str: str):
    """Plan for per-sample response tails.  Sample i scores n_i = lens[i] - lab_shift rows starting at
    sequence position (L_seq - lens[i] + row_shift), against labels lab[i, lab_shift : lens[i]]."""
    device = torch.device(device_str)
    n = len(lens)
    counts = [max(r - lab_shift, 0) for r in lens]
    W = max(counts) if width is None else width
    first = [L_seq - r + row_shift for r in lens]
    return RowPlan(
        [i * sb + first[i] * sl for i in range(n)], [i * lab_stride + lab_shift for i in range(n)],
        [i * W for i in range(n)], counts, [i * L_seq + first[i] for i in range(n)], (n, W), n * L_seq, device,
    )


# ---- K1 / K1b autograd ---------------------------------------------------------------------------
def _launch_fwd(logits, labels, plan: RowPlan, out, stat_max, stat_logsum, ignore_index=None):
    dev = logits.device
    sc = _device_scratch(dev)
    p = plan.ptrs()
    L.check(L.lib().aa_logprob_fwd(
        logits.data_ptr(), L.dtype_code(logits.dtype), logits.stride(-2), logits.size(-1), labels.data_ptr(),
        0 if ignore_index is None else int(ignore_index), 0 if ignore_index is None else 1,
        plan.n_seg, plan.n_rows, p[0], p[1], p[2], p[3], out.data_ptr(), L.dtype_code(out.dtype),
        L.ptr(stat_max), L.ptr(stat_logsum), sc['status'].data_ptr(), L.stream_ptr(dev)))


def _launch_bwd(logits, labels, plan: RowPlan, stat_max, stat_logsum, grad_rows, grad_seg, grad_scale,
                grad_logits, mode_code, scratch=None, ignore_index=None, grad_row_stride=None):
    dev = logits.device
    p = plan.ptrs()
    V = logits.size(-1)
    n_tile_rows, extra, n_extra = plan.n_tile_rows, None, 0
    if n_tile_rows > 0 and _ZERO_SPANS and plan.host_layout:
        # the row layout is known on the host: long zero spans -> copy engine, isolated zero rows -> listed after the
        # scored rows (equal-cost rows first under the kernel's static stride), instead of "every tile row is work"
        import ctypes

        if plan.n_zero_spans:
            L.check(L.lib().aa_zero_rows(grad_logits.data_ptr(), L.dtype_code(grad_logits.dtype), V, V, plan.n_tile_rows,
                                         ctypes.cast(plan.zero_spans, ctypes.c_void_p), plan.n_zero_spans,
                                         L.stream_ptr(dev)))
        n_tile_rows, extra, n_extra = 0, plan.extra_zero_rows, plan.n_extra
    if scratch is None:  # 32 bytes per work row: the RowRec table of the TMA-staged K1b
        n_work = n_tile_rows if n_tile_rows > 0 else plan.n_rows + n_extra
        scratch = torch.empty(max(n_work, 1) * 4, dtype=torch.int64, device=dev)
    L.check(L.lib().aa_logprob_bwd(
        logits.data_ptr(), L.dtype_code(logits.dtype), logits.stride(-2), logits.size(-1), labels.data_ptr(),
        0 if ignore_index is None else int(ignore_index), 0 if ignore_index is None else 1,
        plan.n_seg, plan.n_rows, p[0], p[1], p[2], p[3], p[4], stat_max.data_ptr(), stat_logsum.data_ptr(),
        L.ptr(grad_rows), L.dtype_code(grad_rows.dtype) if grad_rows is not None else L.AA_F32,
        L.ptr(grad_seg), L.ptr(grad_scale), L.dtype_code(grad_scale.dtype) if grad_scale is not None else L.AA_F32,
        grad_logits.data_ptr(), V if grad_row_stride is None else int(grad_row_stride),
        n_tile_rows, L.ptr(extra), n_extra,
        L.ptr(scratch), mode_code, L.stream_ptr(dev)))


class _LogProbFn(torch.autograd.Function):
    """K1 forward / K1b backward.  `logits` is the tensor the gradient tile is shaped after; the plan
    addresses rows inside it."""

    @staticmethod
    def forward(ctx, logits, labels, plan: RowPlan, mode_code: int):
        out_dtype = logits.dtype if mode_code == L.MODE_FAITHFUL else torch.float32
        n_out = 1
        for d in plan.out_shape:
            n_out *= d
        fully_covered = plan.exact and (n_out == plan.n_rows)
        out = (torch.empty if fully_covered else torch.zeros)(plan.out_shape, dtype=out_dtype, device=logits.device)
        need_grad = ctx.needs_input_grad[0]  # grad mode is off inside forward(); this is the apply-time truth
        stat_max = stat_logsum = None
        if need_grad:
            stats = torch.empty((2, max(plan.n_rows, 1)), dtype=torch.float32, device=logits.device)
            stat_max, stat_logsum = stats[0], stats[1]
        _launch_fwd(logits, labels, plan, out, stat_max, stat_logsum)
        if need_grad:
            ctx.save_for_backward(logits, labels, stats)
            ctx.plan = plan
            ctx.mode_code = mode_code
        return out

    @staticmethod
    def backward(ctx, grad_out):
        logits, labels, stats = ctx.saved_tensors
        plan = ctx.plan
        grad_out = grad_out.contiguous()
        if grad_out.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            grad_out = grad_out.float()
        grad = torch.empty(logits.shape, dtype=logits.dtype, device=logits.device)
        _launch_bwd(logits, labels, plan, stats[0], stats[1], grad_out, None, None, grad, ctx.mode_code)
        return grad, None, None, None


def _contiguous_last(t: torch.Tensor) -> torch.Tensor:
    return t if t.stride(-1) == 1 else t.contiguous()


def _try_reroute(logits: torch.Tensor):
    """If `logits` is a row-aligned view of a contiguous base (e.g. `full[:, :-1]`,
    `full[idx][-R:]`), address the BASE instead so the backward writes the base's gradient tile
    directly (zero rows included) and autograd's slice-backward never materialises a padded copy."""
    if not (_REROUTE_TO_BASE and logits._is_view()):
        return None
    base = logits._base
    V = logits.size(-1)
    if base is None or base.dim() < 2 or base.size(-1) != V or not base.is_contiguous():
        return None
    if base.dtype != logits.dtype or logits.stride(-1) != 1 or logits.stride(-2) != V:
        return None
    off = logits.storage_offset() - base.storage_offset()
    if off < 0 or off % V or (logits.dim() == 3 and logits.stride(0) % V):
        return None
    return base, off // V


def gather_log_probabilities(logits: torch.Tensor, labels: torch.Tensor, mode: str | None = None) -> torch.Tensor:
    """Drop-in for utils/tools.py:402-413: log_softmax(logits, -1) gathered at `labels`, without ever
    writing the (B, L, V) log-prob tile.  logits (B, L, V) or (L, V), any batch/row strides (the
    callers pass `[:, :-1]` views); differentiable in `logits` (K1b)."""
    L.require_cuda(logits, labels)
    squeeze = logits.dim() == 2
    if squeeze:
        logits, labels = logits.unsqueeze(0), labels.unsqueeze(0)
    if logits.dim() != 3 or labels.shape != logits.shape[:2]:
        raise ValueError(f'expected logits (B, L, V) and labels (B, L); got {tuple(logits.shape)}, {tuple(labels.shape)}')
    logits = _contiguous_last(logits)
    if labels.dtype != torch.int64:
        labels = labels.to(torch.int64)
    labels = _contiguous_last(labels)
    B, rows, V = logits.shape
    mode_code = _mode_code(mode, logits.dtype)
    dev = str(logits.device)
    if B == 0 or rows == 0:
        out_dtype = logits.dtype if mode_code == L.MODE_FAITHFUL else torch.float32
        out = logits.new_zeros((B, rows), dtype=out_dtype)
        return out.squeeze(0) if squeeze else out
    routed = _try_reroute(logits) if (logits.requires_grad and torch.is_grad_enabled()) else None
    lab_sb = labels.stride(0) if B > 1 else rows
    if routed is not None:
        base, row0 = routed
        n_tile = base.numel() // V
        sb_rows = logits.stride(0) // V if B > 1 else rows
        # logits offsets in the plan are relative to the view's first row (row0 of the base); tile rows are
        # rows of the base, whose shape the gradient takes
        plan = _dense_plan(B, rows, sb_rows * V, V, lab_sb, row0, sb_rows, n_tile, dev)
        out = _LogProbViewFn.apply(base, row0, labels, plan, mode_code)
    else:
        sb = logits.stride(0) if B > 1 else rows * logits.stride(1)
        plan = _dense_plan(B, rows, sb, logits.stride(1), lab_sb, 0, rows, B * rows, dev)
        out = _LogProbFn.apply(logits, labels, plan, mode_code)
    return out.squeeze(0) if squeeze else out


# ---- lm_head x log-prob without the (rows, V) tile (SURVEY.md 8f rank 1, first step) ------------------------
def _mm_f32(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """a @ b with an fp32 result (cuBLAS accumulates in fp32 anyway; this keeps the accumulator's precision)."""
    if a.dtype == torch.float32:
        return torch.mm(a, b)
    try:
        return torch.mm(a, b, out_dtype=torch.float32)
    except (TypeError, NotImplementedError, RuntimeError):  # no mixed-dtype mm: one rounding per chunk
        return torch.mm(a, b).float()


def _pad_vocab(weight: torch.Tensor):
    """Weight with the vocabulary padded (zero rows) to a 16-byte multiple of logits per row.  V = 128257 is odd: a
    (rows, V) logits buffer then has 2-byte aligned rows, cuBLAS falls back to its unaligned kernels (measured
    124 TFLOP/s instead of ~1400 on B200) and K1 / K1b lose their 16-byte fast paths."""
    V, H = weight.shape
    q = 16 // weight.element_size()
    Vp = (V + q - 1) // q * q
    if Vp == V:
        return weight, V
    w = torch.zeros((Vp, H), dtype=weight.dtype, device=weight.device)
    w[:V].copy_(weight)
    return w, Vp


class _LinearLogProbFn(torch.autograd.Function):
    """log_softmax(hidden @ weight.T)[label] per row, `chunk` rows at a time: the GEMM (cuBLAS through
    torch.matmul -- a plain library GEMM, on a vocabulary-padded copy of the weight so that every leading dimension
    is 16-byte aligned) writes a (chunk, V_pad) buffer that K1 consumes immediately and the next chunk overwrites;
    the backward recomputes the chunk, K1b turns it into d(logits) in a second buffer (pad columns stay zero), and
    two more GEMMs accumulate d(hidden) and d(weight).  Only (max, log-sum) per row is saved.  HBM held: 2 chunk
    buffers, the padded weight and an fp32 d(weight) accumulator instead of two (rows, V) tiles."""

    @staticmethod
    def forward(ctx, hidden, weight, labels, chunk: int, mode_code: int):
        N, V = hidden.size(0), weight.size(0)
        dev = hidden.device
        out_dtype = hidden.dtype if mode_code == L.MODE_FAITHFUL else torch.float32
        out = torch.empty(N, dtype=out_dtype, device=dev)
        need_grad = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        stats = torch.empty((2, max(N, 1)), dtype=torch.float32, device=dev) if need_grad else None
        w_pad, Vp = _pad_vocab(weight)
        buf = torch.empty((min(chunk, N), Vp), dtype=hidden.dtype, device=dev)
        for r0 in range(0, N, chunk):
            n = min(chunk, N - r0)
            torch.matmul(hidden[r0:r0 + n], w_pad.t(), out=buf[:n])  # the dtype rounding point of nn.Linear
            plan = _dense_plan(1, n, n * Vp, Vp, n, 0, n, 0, str(dev))
            _launch_fwd(buf[:n, :V], labels[r0:r0 + n], plan, out[r0:r0 + n],
                        stats[0, r0:r0 + n] if need_grad else None, stats[1, r0:r0 + n] if need_grad else None)
        if need_grad:
            ctx.save_for_backward(hidden, weight, labels, stats)
            ctx.chunk, ctx.mode_code = chunk, mode_code
        return out

    @staticmethod
    def backward(ctx, grad_out):
        hidden, weight, labels, stats = ctx.saved_tensors
        N, V, chunk = hidden.size(0), weight.size(0), ctx.chunk
        dev = hidden.device
        grad_out = grad_out.contiguous()
        if grad_out.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            grad_out = grad_out.float()
        need_h, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        w_pad, Vp = _pad_vocab(weight)
        d_hidden = torch.empty_like(hidden) if need_h else None
        d_weight = torch.zeros((Vp, weight.size(1)), dtype=torch.float32, device=dev) if need_w else None
        buf = torch.empty((min(chunk, N), Vp), dtype=hidden.dtype, device=dev)
        dbuf = torch.zeros_like(buf)  # K1b writes columns [0, V); the pad columns must stay 0 for the GEMMs below
        for r0 in range(0, N, chunk):
            n = min(chunk, N - r0)
            torch.matmul(hidden[r0:r0 + n], w_pad.t(), out=buf[:n])
            plan = _dense_plan(1, n, n * Vp, Vp, n, 0, n, 0, str(dev))
            _launch_bwd(buf[:n, :V], labels[r0:r0 + n], plan, stats[0, r0:r0 + n], stats[1, r0:r0 + n],
                        grad_out[r0:r0 + n], None, None, dbuf[:n, :V], ctx.mode_code, grad_row_stride=Vp)
            if need_h:
                torch.matmul(dbuf[:n], w_pad, out=d_hidden[r0:r0 + n])
            if need_w:  # fp32 accumulation across chunks, one rounding at the end (like a single GEMM)
                d_weight.add_(_mm_f32(dbuf[:n].t(), hidden[r0:r0 + n]))
        return d_hidden, (d_weight[:V].to(weight.dtype) if need_w else None), None, None, None


class _LinearLogProbK6Fn(torch.autograd.Function):
    """The tensor-core path (bf16, H % 64 == 0; default).  Forward = K6 (no logits at all, saves (max, logsum) per row).
    Backward per row chunk = three tcgen05 kernels on one (chunk, ld) bf16 d(logits) buffer: K6b recomputes the logits
    tile and turns it into d(logits) in its epilogue; aa_linear_dhidden = d(logits) @ W with W consumed MN-major in
    place; aa_linear_dweight accumulates d(logits)^T @ hidden in fp32 across chunks and rounds once at the end.  No
    library GEMM, no padded / transposed copy of the weight."""

    @staticmethod
    def forward(ctx, hidden, weight, labels, chunk: int, mode_code: int):
        out, stats = fused_linear_token_log_probs(hidden, weight, labels, _K6_MODE_NAME[mode_code], return_stats=True)
        ctx.save_for_backward(hidden, weight, labels, stats)
        ctx.chunk, ctx.mode_code = chunk, mode_code
        return out

    @staticmethod
    def backward(ctx, grad_out):
        hidden, weight, labels, stats = ctx.saved_tensors
        N, (V, H), chunk = hidden.size(0), weight.shape, ctx.chunk
        dev = hidden.device
        grad_out = grad_out.contiguous()
        if grad_out.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            grad_out = grad_out.float()
        ld = (V + 255) // 256 * 256
        need_h, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        d_hidden = torch.empty_like(hidden) if need_h else None
        d_weight = torch.empty_like(weight) if need_w else None
        n_chunks = (N + chunk - 1) // chunk
        # equal chunks of whole 256-row CTA-pair tiles: 16376 rows as 8192 + 8184 keep the last round of 256 x 256 tiles of
        # the d(hidden) GEMM full (512 tiles on 74 pairs = 6.9 rounds), 8320 + 8056 does not (528 tiles = 7.1 rounds run as 8)
        chunk = min(chunk, (-(-N // n_chunks) + 255) // 256 * 256)
        acc = torch.empty((V, H), dtype=torch.float32, device=dev) if (need_w and n_chunks > 1) else None
        dbuf = torch.empty((min(chunk, N), ld), dtype=torch.bfloat16, device=dev)
        lib, st = L.lib(), L.stream_ptr(dev)
        for i, r0 in enumerate(range(0, N, chunk)):
            n = min(chunk, N - r0)
            h = hidden[r0:r0 + n]
            L.check(lib.aa_linear_dlogits(
                h.data_ptr(), n, H, h.stride(0), weight.data_ptr(), V, weight.stride(0), labels[r0:r0 + n].data_ptr(),
                stats[0, r0:r0 + n].data_ptr(), stats[1, r0:r0 + n].data_ptr(), grad_out[r0:r0 + n].data_ptr(),
                L.dtype_code(grad_out.dtype), dbuf.data_ptr(), ld, ctx.mode_code, st))
            if need_h:
                dh = d_hidden[r0:r0 + n]
                L.check(lib.aa_linear_dhidden(dbuf.data_ptr(), n, ld, weight.data_ptr(), V, H, weight.stride(0),
                                              dh.data_ptr(), dh.stride(0), st))
            if need_w:
                last = i == n_chunks - 1
                L.check(lib.aa_linear_dweight(dbuf.data_ptr(), n, ld, h.data_ptr(), H, h.stride(0), V, L.ptr(acc), H,
                                              1 if i > 0 else 0, d_weight.data_ptr() if last else None, d_weight.stride(0), st))
        return d_hidden, d_weight, None, None, None


_K6_MODE_NAME = {L.MODE_FAITHFUL: 'faithful', L.MODE_F32: 'f32', L.MODE_CE: 'ce'}


def linear_token_log_probs(hidden: torch.Tensor, weight: torch.Tensor, labels: torch.Tensor,
                           chunk_rows: int | None = None, mode: str | None = None) -> torch.Tensor:
    """gather_log_probabilities(F.linear(hidden, weight), labels) for hidden (N, H), weight (V, H), labels (N,)
    without materialising the (N, V) logits / gradient tiles.  Differentiable in hidden and weight.
    mode='ce': the rounding of a cross-entropy on `F.linear(hidden, weight).float()` -- logits rounded to the operand
    dtype (nn.Linear's output), fp32 log-probs, d(logits) rounded once."""
    L.require_cuda(hidden, weight, labels)
    if hidden.dim() != 2 or weight.dim() != 2 or hidden.size(1) != weight.size(1) or labels.shape != hidden.shape[:1]:
        raise ValueError('expected hidden (N, H), weight (V, H), labels (N,)')
    if hidden.dtype != weight.dtype:
        raise ValueError('hidden and weight must share a dtype')
    V = weight.size(0)
    if hidden.size(0) == 0:
        return hidden.new_zeros((0,))
    labels = labels.to(torch.int64).contiguous()
    if _K6B and hidden.dtype == torch.bfloat16 and hidden.size(1) % 64 == 0:
        if chunk_rows is None:  # ~2 GB of d(logits) per chunk: few read-modify-write passes over the fp32 d(weight)
            chunk_rows = max(128, (2 << 30) // ((V + 255) // 256 * 256 * 2) // 128 * 128)
        return _LinearLogProbK6Fn.apply(hidden.contiguous(), weight.contiguous(), labels, int(chunk_rows),
                                        L.MODE_CE if mode == 'ce' else _mode_code(mode, hidden.dtype))
    # f16 / f32 operands or H % 64 != 0: library GEMMs (cuBLAS) around K1 / K1b -- not the product's hot configuration
    if chunk_rows is None:  # ~256 MB of logits per chunk
        chunk_rows = max(128, (256 << 20) // (V * hidden.element_size()) // 128 * 128)
    return _LinearLogProbFn.apply(hidden.contiguous(), weight.contiguous(), labels, int(chunk_rows),
                                  L.MODE_F32 if mode == 'ce' else _mode_code(mode, hidden.dtype))


def fused_linear_token_log_probs(hidden: torch.Tensor, weight: torch.Tensor, labels: torch.Tensor,
                                 mode: str | None = None, return_stats: bool = False):
    """K6 (tcgen05): log_softmax(hidden @ weight.T)[label] per row in ONE kernel, no logits tile, for rows that
    carry NO gradient (reference model / rollout scoring).  hidden (N, H) bf16, weight (V, H) bf16, H % 64 == 0."""
    L.require_cuda(hidden, weight, labels)
    if hidden.dim() != 2 or weight.dim() != 2 or hidden.size(1) != weight.size(1) or labels.shape != hidden.shape[:1]:
        raise ValueError('expected hidden (N, H), weight (V, H), labels (N,)')
    if hidden.dtype != torch.bfloat16 or weight.dtype != torch.bfloat16:
        raise ValueError('K6 takes bf16 operands')
    hidden, weight = _contiguous_last(hidden.detach()), _contiguous_last(weight.detach())
    labels = labels.to(torch.int64).contiguous()
    N, V = hidden.size(0), weight.size(0)
    mode_code = L.MODE_CE if mode == 'ce' else _mode_code(mode, hidden.dtype)
    out = torch.empty(N, dtype=torch.bfloat16 if mode_code == L.MODE_FAITHFUL else torch.float32, device=hidden.device)
    stats = torch.empty((2, max(N, 1)), dtype=torch.float32, device=hidden.device) if return_stats else None
    sc = _device_scratch(hidden.device)
    partial = torch.empty(3 * max(148 * 128, 16 * N), dtype=torch.float32, device=hidden.device)  # split-vocabulary statistics
    L.check(L.lib().aa_linear_logprob_fwd(
        hidden.data_ptr(), N, hidden.size(1), hidden.stride(0), weight.data_ptr(), V, weight.stride(0), labels.data_ptr(),
        out.data_ptr(), L.dtype_code(out.dtype), L.ptr(stats[0]) if return_stats else None,
        L.ptr(stats[1]) if return_stats else None, partial.data_ptr(), partial.numel(), mode_code,
        sc['status'].data_ptr(), L.stream_ptr(hidden.device)))
    return (out, stats) if return_stats else out


def lm_head_weight(module) -> torch.Tensor:
    """The (V, H) weight of a causal LM's output head for the fused lm_head paths, or a clear error where those paths
    would be silently wrong: the weight is used OUTSIDE the module's forward, so it must be materialised here (under
    DeepSpeed ZeRO-3 it is a partitioned placeholder), and the head must be a plain bias-free projection of
    `hidden_states[-1]` without logit scaling / soft-capping (Gemma-2, Cohere)."""
    head = module.get_output_embeddings()
    weight = head.weight
    if hasattr(weight, 'ds_id') or weight.numel() == 0:
        raise RuntimeError('fused_lm_head is not supported under DeepSpeed ZeRO-3: the lm_head weight is partitioned outside '
                           'the module forward (use the default logits-tile path, or ZeRO <= 2)')
    if getattr(head, 'bias', None) is not None:
        raise RuntimeError('fused_lm_head needs a bias-free lm_head')
    cfg = getattr(module, 'config', None)
    for key in ('final_logit_softcapping', 'logit_scale'):
        if getattr(cfg, key, None) not in (None, 1.0):
            raise RuntimeError(f'fused_lm_head does not reproduce `{key}` = {getattr(cfg, key)}: use the default logits-tile path')
    if weight.dim() != 2:
        raise RuntimeError('fused_lm_head expects a (V, H) head weight')
    return weight


@functools.lru_cache(maxsize=64)
def _tail_indices(counts: tuple, first_pos: tuple, seq: int, W: int, device_str: str):
    """Host-built (cached, copied once) gather / scatter indices of the scored rows: flat position i * seq + first_i + k in
    the (n * seq, H) hidden matrix and i * W + k in the padded (n, W) output, k < counts_i.  The counts are host values
    (the callers hold the response lengths as Python ints), so no boolean indexing and no device->host sync is needed."""
    src, dst = [], []
    for i, (c, f) in enumerate(zip(counts, first_pos)):
        for k in range(max(int(c), 0)):
            src.append(i * seq + min(max(int(f) + k, 0), seq - 1))
            dst.append(i * W + k)
    dev = torch.device(device_str)
    return (torch.tensor(src, dtype=torch.int64).to(dev, non_blocking=True),
            torch.tensor(dst, dtype=torch.int64).to(dev, non_blocking=True))


def _tails_from_hidden(hidden, weight, labels_padded, lens, counts, first_pos, lab_shift, chunk_rows, mode):
    """Sample i scores counts[i] rows: hidden position first_pos[i] + k against labels_padded[i, lab_shift + k].
    The scored rows are gathered into a compact (rows, H) matrix: K6 when nothing needs a gradient, else K6 + K6b + the
    two backward GEMMs (linear_token_log_probs).  Returns (n, max(counts)) right-padded with 0."""
    n, seq, H = hidden.shape
    W = max(max(counts), 0)
    out_dtype = hidden.dtype if _mode_code(mode, hidden.dtype) == L.MODE_FAITHFUL else torch.float32
    if W == 0:
        return hidden.new_zeros((n, 0), dtype=out_dtype)
    dev = hidden.device
    src, dst = _tail_indices(tuple(int(c) for c in counts), tuple(int(f) for f in first_pos), seq, W, str(dev))
    rows = hidden.reshape(n * seq, H).index_select(0, src)
    lab = labels_padded[:, lab_shift:lab_shift + W].reshape(-1).index_select(0, dst)
    needs_grad = torch.is_grad_enabled() and (hidden.requires_grad or weight.requires_grad)
    if not needs_grad and _K6 and hidden.dtype == torch.bfloat16 and weight.dtype == torch.bfloat16 and H % 64 == 0:
        lp = fused_linear_token_log_probs(rows, weight, lab, mode)  # K6: one tcgen05 kernel, no logits at all
    else:
        lp = linear_token_log_probs(rows, weight, lab, chunk_rows, mode)
    return torch.zeros(n * W, dtype=lp.dtype, device=dev).index_copy(0, dst, lp).view(n, W)


def sequence_log_probs_from_hidden(hidden: torch.Tensor, weight: torch.Tensor, input_ids: torch.Tensor,
                                   response_lens: Sequence[int], pad_id: int, strip: bool = True,
                                   chunk_rows: int | None = None, mode: str | None = None) -> torch.Tensor:
    """DPOTrainer.compute_log_probs (trainers/text_to_text/dpo.py:122-142) from the LAST HIDDEN STATES
    (2B, L, H) and the lm_head weight (V, H): the scored rows are gathered into a compact (rows, H) matrix and
    go through K6 / linear_token_log_probs, so no (2B, L, V) tile exists in either direction."""
    L.require_cuda(hidden, weight, input_ids)
    lens = tuple(int(r) for r in response_lens)
    seq = hidden.size(1)
    labels = strip_pad_tail(input_ids, lens, pad_id, strip)  # (n, max R); row i scores labels[i, 1:R_i]
    return _tails_from_hidden(hidden, weight, labels, lens, [max(r - 1, 0) for r in lens], [seq - r for r in lens], 1,
                              chunk_rows, mode)


def tail_log_probs_from_hidden(hidden: torch.Tensor, weight: torch.Tensor, input_ids: torch.Tensor,
                               response_lens: Sequence[int], chunk_rows: int | None = None,
                               mode: str | None = None) -> torch.Tensor:
    """The multimodal PPO scoring rows (trainers/text_image_to_text/ppo.py:233-246, 296-309): sample b scores
    `logits[b, :-1][-R_b:]` against `input_ids[b, 1:][-R_b:]`, here from the last hidden states (B, L, H) and the
    lm_head weight -- hidden position L - 1 - R_b + k predicts token L - R_b + k."""
    L.require_cuda(hidden, weight, input_ids)
    lens = tuple(int(r) for r in response_lens)
    seq = hidden.size(1)
    labels = strip_pad_tail(input_ids, lens, 0, strip=False)  # (B, max R): input_ids[b, -R_b:]
    return _tails_from_hidden(hidden, weight, labels, lens, list(lens), [seq - 1 - r for r in lens], 0, chunk_rows, mode)


class _LogProbViewFn(torch.autograd.Function):
    """Same as _LogProbFn but the differentiable input is the contiguous BASE tensor of the view the caller
    passed; the scored rows start at row `first_row` of the base viewed as (rows, V)."""

    @staticmethod
    def forward(ctx, base, first_row: int, labels, plan: RowPlan, mode_code: int):
        V = base.size(-1)
        view = base.view(-1, V)[first_row:]
        out_dtype = base.dtype if mode_code == L.MODE_FAITHFUL else torch.float32
        out = torch.empty(plan.out_shape, dtype=out_dtype, device=base.device)
        stats = torch.empty((2, plan.n_rows), dtype=torch.float32, device=base.device)
        _launch_fwd(view, labels, plan, out, stats[0], stats[1])
        ctx.save_for_backward(base, labels, stats)
        ctx.plan, ctx.mode_code, ctx.first_row = plan, mode_code, first_row
        return out

    @staticmethod
    def backward(ctx, grad_out):
        base, labels, stats = ctx.saved_tensors
        V = base.size(-1)
        view = base.view(-1, V)[ctx.first_row:]
        grad_out = grad_out.contiguous()
        if grad_out.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            grad_out = grad_out.float()
        grad = torch.empty(base.shape, dtype=base.dtype, device=base.device)
        _launch_bwd(view, labels, ctx.plan, stats[0], stats[1], grad_out, None, None, grad, ctx.mode_code)
        return grad, None, None, None, None


# ---- DPO -----------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=64)
def _lens_tensor(lens: tuple, device_str: str):
    return torch.tensor(lens, dtype=torch.int32).to(device_str, non_blocking=True)


def strip_pad_tail(input_ids: torch.Tensor, response_lens: Sequence[int], pad_id: int, strip: bool = True):
    """labels[i, :R_i] = strip_pad(input_ids[i])[-R_i:] (trainers/text_to_text/dpo.py:52-54,135-137),
    or the plain tail input_ids[i, -R_i:] when strip=False (text_audio_to_text/dpo.py:100).
    Returns an int64 (n, max R) buffer (entries beyond R_i undefined)."""
    L.require_cuda(input_ids)
    lens = tuple(int(r) for r in response_lens)
    n, seq = input_ids.shape
    if len(lens) != n:
        raise ValueError('response_lens must have one entry per row of input_ids')
    if min(lens) < 1 or max(lens) > seq:
        raise ValueError(f'response_lens must lie in [1, {seq}]; got {lens}')
    input_ids = _contiguous_last(input_ids)
    out = torch.empty((n, max(lens)), dtype=torch.int64, device=input_ids.device)
    sc = _device_scratch(input_ids.device)
    L.check(L.lib().aa_strip_pad_tail(
        input_ids.data_ptr(), n, seq, input_ids.stride(0), int(pad_id), 1 if strip else 0,
        _lens_tensor(lens, str(input_ids.device)).data_ptr(), out.data_ptr(), out.stride(0),
        sc['status'].data_ptr(), L.stream_ptr(input_ids.device)))
    return out


def _dpo_plan(logits: torch.Tensor, lens: tuple, label_stride: int):
    n, seq, V = logits.shape
    if logits.stride(-1) != 1:
        raise ValueError('logits must be contiguous in the vocab dimension')
    return _tail_plan(lens, seq, logits.stride(0), logits.stride(1), label_stride, 1, 0, None, str(logits.device))


def sequence_log_probs(logits: torch.Tensor, input_ids: torch.Tensor, response_lens: Sequence[int], pad_id: int,
                       strip: bool = True, mode: str | None = None) -> torch.Tensor:
    """The arithmetic of DPOTrainer.compute_log_probs after the model forward
    (trainers/text_to_text/dpo.py:129-142; text_image_to_text/dpo.py:92-105; strip=False:
    text_audio_to_text/dpo.py:93-105): for sample i the R_i - 1 log-probs of its response tail,
    right-padded with 0 to max(R) - 1.  ONE launch for all samples, no host sync."""
    L.require_cuda(logits, input_ids)
    lens = tuple(int(r) for r in response_lens)
    labels = strip_pad_tail(input_ids, lens, pad_id, strip)
    logits = _contiguous_last(logits)
    plan = _dpo_plan(logits, lens, labels.stride(0))
    return _LogProbFn.apply(logits, labels, plan, _mode_code(mode, logits.dtype))


def _dpo_launch(policy_lp, ref_lp, scale_coeff, mode_code, input_ids, want_grad_seg, coll=None):
    """coll: an `_lib.AaColl` descriptor (utils.multi_process.FusedPackedAllReduce.next()) -> K2's last block
    also all-reduces the stats over NVLink; the reduced vector comes back as a 4th result."""
    import ctypes

    dev = policy_lp.device
    n2, W = policy_lp.shape
    B = n2 // 2
    per_pair = torch.empty((5, B), dtype=torch.float32, device=dev)
    stats = torch.empty(8, dtype=torch.float32, device=dev)
    grad_seg = torch.empty(n2, dtype=torch.float32, device=dev) if want_grad_seg else None
    sc = _device_scratch(dev)
    ids = None
    if input_ids is not None:
        ids = _contiguous_last(input_ids)
    stats_global = torch.empty(8, dtype=torch.float32, device=dev) if coll is not None else None
    L.check(L.lib().aa_dpo_loss(
        policy_lp.data_ptr(), ref_lp.data_ptr(), L.dtype_code(policy_lp.dtype), B, W, policy_lp.stride(0),
        float(scale_coeff), mode_code, L.ptr(ids), ids.size(1) if ids is not None else 0,
        ids.stride(0) if ids is not None else 0, per_pair.data_ptr(), L.ptr(grad_seg), stats.data_ptr(),
        sc['counter'][0:1].data_ptr(), ctypes.byref(coll) if coll is not None else None, L.ptr(stats_global),
        sc['status'].data_ptr(), L.stream_ptr(dev)))
    if coll is not None:
        return per_pair, stats, grad_seg, stats_global
    return per_pair, stats, grad_seg


def _dpo_dict(per_pair, stats, out_dtype, skip_identical):
    loss_i, better, worse, _, valid = per_pair
    if skip_identical:  # the reference stacks only the kept pairs (data-dependent shape -> one sync)
        keep = valid.bool()
        better, worse = better[keep], worse[keep]
    better = better.to(out_dtype)
    worse = worse.to(out_dtype)
    return {
        'reward': better + worse,
        'better_sample_reward': better,
        'worse_sample_reward': worse,
        'reward_accuracy': stats[4],
        'reward_margin': better - worse,
    }


class _DpoFromLpFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, policy_lp, ref_lp, scale_coeff, mode_code, input_ids):
        per_pair, stats, grad_seg = _dpo_launch(policy_lp, ref_lp, scale_coeff, mode_code, input_ids, True)
        ctx.save_for_backward(grad_seg)
        ctx.lp_shape, ctx.lp_dtype = policy_lp.shape, policy_lp.dtype
        ctx.mark_non_differentiable(per_pair, stats)
        out_dtype = policy_lp.dtype if mode_code == L.MODE_FAITHFUL else torch.float32
        return stats[0].to(out_dtype), per_pair, stats

    @staticmethod
    def backward(ctx, g_loss, _g1, _g2):
        (grad_seg,) = ctx.saved_tensors
        g = (grad_seg * g_loss.float()).to(ctx.lp_dtype)
        return g.unsqueeze(1).expand(ctx.lp_shape), None, None, None, None


def dpo_loss_from_log_probs(policy_lp: torch.Tensor, ref_lp: torch.Tensor, scale_coeff: float,
                            input_ids: torch.Tensor | None = None, skip_identical_pairs: bool = False,
                            mode: str | None = None) -> dict[str, torch.Tensor]:
    """trainers/text_to_text/dpo.py:150-203 given the two (2B, W) log-prob tensors: ONE launch for
    the 4 sums per pair, the log-sigmoid loss and the five metrics (K2).  `skip_identical_pairs`:
    text_audio_to_text/dpo.py:134-139.  Extra key '_stats' = packed fp32[8] local means for
    the all-reduce (utils.multi_process.all_reduce_packed)."""
    L.require_cuda(policy_lp, ref_lp)
    if policy_lp.shape != ref_lp.shape or policy_lp.dim() != 2 or policy_lp.size(0) % 2:
        raise ValueError('policy / reference log-probs must both be (2B, W)')
    policy_lp = policy_lp if policy_lp.stride(1) == 1 or policy_lp.size(1) <= 1 else policy_lp.contiguous()
    ref_lp = ref_lp.to(policy_lp.dtype).contiguous()
    if policy_lp.stride(0) != ref_lp.stride(0):
        policy_lp = policy_lp.contiguous()
    mode_code = _mode_code(mode, policy_lp.dtype)
    ids = input_ids if skip_identical_pairs else None
    loss, per_pair, stats = _DpoFromLpFn.apply(policy_lp, ref_lp.detach(), scale_coeff, mode_code, ids)
    out_dtype = policy_lp.dtype if mode_code == L.MODE_FAITHFUL else torch.float32
    out = {'loss': loss}
    out.update(_dpo_dict(per_pair, stats, out_dtype, skip_identical_pairs))
    out['_stats'] = stats
    out['_per_pair'] = per_pair
    return out


class _DpoFusedFn(torch.autograd.Function):
    """policy logits (grad) + reference logits (no grad) -> DPO loss.  Forward: K1 x2, K2.  Backward:
    ONE K1b launch taking the per-sample coefficient straight from K2 (no per-row gradient tensor)."""

    @staticmethod
    def forward(ctx, policy_logits, ref_logits, labels, plan, scale_coeff, mode_code, ids, coll=None):
        dev = policy_logits.device
        out_dtype = policy_logits.dtype if mode_code == L.MODE_FAITHFUL else torch.float32
        lp = torch.zeros((2,) + plan.out_shape, dtype=out_dtype, device=dev)
        need_grad = ctx.needs_input_grad[0]
        stats_rows = torch.empty((2, max(plan.n_rows, 1)), dtype=torch.float32, device=dev) if need_grad else None
        _launch_fwd(policy_logits, labels, plan, lp[0], stats_rows[0] if need_grad else None,
                    stats_rows[1] if need_grad else None)
        _launch_fwd(ref_logits, labels, plan, lp[1], None, None)
        res = _dpo_launch(lp[0], lp[1], scale_coeff, mode_code, ids, True, coll)
        per_pair, stats, grad_seg = res[0], res[1], res[2]
        stats_global = res[3] if coll is not None else stats
        if need_grad:
            ctx.save_for_backward(policy_logits, labels, stats_rows, grad_seg)
            ctx.plan, ctx.mode_code = plan, mode_code
        ctx.mark_non_differentiable(per_pair, stats, lp, stats_global)
        return stats[0].to(out_dtype), per_pair, stats, lp, stats_global

    @staticmethod
    def backward(ctx, g_loss, *_):
        logits, labels, stats_rows, grad_seg = ctx.saved_tensors
        grad = torch.empty(logits.shape, dtype=logits.dtype, device=logits.device)
        scale = g_loss.detach().to(torch.float32).reshape(1).contiguous()
        _launch_bwd(logits, labels, ctx.plan, stats_rows[0], stats_rows[1], None, grad_seg, scale, grad,
                    ctx.mode_code)
        return grad, None, None, None, None, None, None, None


def dpo_fused_loss(policy_logits: torch.Tensor, ref_logits: torch.Tensor, input_ids: torch.Tensor,
                   response_lens: Sequence[int], pad_id: int, scale_coeff: float, strip: bool = True,
                   skip_identical_pairs: bool = False, mode: str | None = None, coll=None) -> dict[str, torch.Tensor]:
    """The whole of DPOTrainer.loss after the two model forwards (trainers/text_to_text/dpo.py:144-203):
    5 launches forward (label extraction, K1 policy, K1 reference, K2), 1 launch backward (K1b)."""
    L.require_cuda(policy_logits, ref_logits, input_ids)
    if policy_logits.shape != ref_logits.shape or policy_logits.dim() != 3:
        raise ValueError('policy / reference logits must both be (2B, L, V)')
    if policy_logits.size(0) % 2 or policy_logits.size(0) != len(response_lens):
        raise ValueError('need 2B rows (chosen first, rejected second) and one response_len per row')
    lens = tuple(int(r) for r in response_lens)
    labels = strip_pad_tail(input_ids, lens, pad_id, strip)
    policy_logits = _contiguous_last(policy_logits)
    ref_logits = ref_logits.detach()
    if ref_logits.stride() != policy_logits.stride() or ref_logits.dtype != policy_logits.dtype:
        ref_logits = ref_logits.to(policy_logits.dtype).contiguous()
        if ref_logits.stride() != policy_logits.stride():
            policy_logits = policy_logits.contiguous()
    plan = _dpo_plan(policy_logits, lens, labels.stride(0))
    mode_code = _mode_code(mode, policy_logits.dtype)
    ids = input_ids if skip_identical_pairs else None
    loss, per_pair, stats, lp, stats_global = _DpoFusedFn.apply(policy_logits, ref_logits, labels, plan, scale_coeff,
                                                               mode_code, ids, coll)
    out_dtype = policy_logits.dtype if mode_code == L.MODE_FAITHFUL else torch.float32
    out = {'loss': loss}
    out.update(_dpo_dict(per_pair, stats, out_dtype, skip_identical_pairs))
    out['_stats'] = stats
    if coll is not None:
        out['_stats_global'] = stats_global  # already averaged over the ranks by K2 itself (NVLink peer memory)
    out['_per_pair'] = per_pair
    out['_log_probs'] = lp
    return out


# ---- SimPO / ORPO / KTO pair bookkeeping ---------------------------------------------------------------
def pair_slices(input_ids: torch.Tensor, attention_mask: torch.Tensor) -> torch.Tensor:
    """trainers/text_to_text/simpo.py:61-77 for all pairs in one launch: int32 (4, B) = valid, diverge_index,
    end_better, end_worse (the reference: a Python loop with 4 host syncs per pair)."""
    L.require_cuda(input_ids, attention_mask)
    n, seq = input_ids.shape
    if n % 2 or attention_mask.shape != input_ids.shape:
        raise ValueError('input_ids / attention_mask must both be (2B, L)')
    ids = _contiguous_last(input_ids)
    mask = attention_mask
    kind = L.MASK_U8
    if mask.dtype == torch.int64:
        kind = L.MASK_I64
    elif mask.dtype != torch.bool:
        mask = mask != 0
    mask = _contiguous_last(mask)
    out = torch.empty((4, n // 2), dtype=torch.int32, device=ids.device)
    sc = _device_scratch(ids.device)
    L.check(L.lib().aa_pair_slices(ids.data_ptr(), ids.stride(0), mask.data_ptr(), kind, mask.stride(0), n // 2, seq,
                                   out.data_ptr(), sc['status'].data_ptr(), L.stream_ptr(ids.device)))
    return out


class _SliceSumFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, lp, slices, mode_code):
        n, W = lp.shape
        sums = torch.empty(n, dtype=torch.float32, device=lp.device)
        L.check(L.lib().aa_slice_sums(lp.data_ptr(), L.dtype_code(lp.dtype), lp.stride(0), n // 2, W, slices.data_ptr(),
                                      mode_code, sums.data_ptr(), L.stream_ptr(lp.device)))
        ctx.save_for_backward(slices)
        ctx.W, ctx.dtype = W, lp.dtype
        return sums.to(lp.dtype) if mode_code == L.MODE_FAITHFUL else sums

    @staticmethod
    def backward(ctx, g):
        (slices,) = ctx.saved_tensors
        B = slices.size(1)
        cols = torch.arange(ctx.W, device=g.device).unsqueeze(0)
        lo = slices[1].repeat(2).unsqueeze(1)
        hi = torch.cat([slices[2], slices[3]]).unsqueeze(1) + 1
        inside = (cols >= lo) & (cols < hi)
        return torch.where(inside, g.unsqueeze(1).to(ctx.dtype), torch.zeros((), dtype=ctx.dtype, device=g.device)), None, None


def slice_sums(sequence_log_probs: torch.Tensor, slices: torch.Tensor, mode: str | None = None) -> torch.Tensor:
    """sum(lp[r, diverge : end + 1]) for the 2B rows (simpo.py:78-79), one launch; differentiable in lp."""
    L.require_cuda(sequence_log_probs, slices)
    lp = _contiguous_last(sequence_log_probs)
    return _SliceSumFn.apply(lp, slices.contiguous(), _mode_code(mode, lp.dtype))


# ---- GRPO ---------------------------------------------------------------------------------------------
def group_advantages(rewards: torch.Tensor, num_generations: int) -> torch.Tensor:
    """trainers/text_to_text/grpo.py:268-274: rewards (B * G,) fp32 -> advantages (B * G, 1),
    (r - group mean) / (unbiased group std + 1e-4)."""
    L.require_cuda(rewards)
    r = rewards.detach().float().contiguous().view(-1)
    if r.numel() % num_generations:
        raise ValueError('rewards must hold B * num_generations values')
    adv = torch.empty_like(r)
    L.check(L.lib().aa_group_advantages(r.data_ptr(), r.numel() // num_generations, int(num_generations), adv.data_ptr(),
                                        L.stream_ptr(r.device)))
    return adv.view(-1, 1)


class _GrpoLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, lp, ref_lp, adv, tokens, eos_id, beta, mode_code):
        B, K = lp.shape
        dev = lp.device
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        grad = torch.empty((B, K), dtype=lp.dtype, device=dev)
        row_end = torch.empty(B, dtype=torch.int32, device=dev)
        scratch = torch.empty(B + 1, dtype=torch.float32, device=dev)
        sc = _device_scratch(dev)
        L.check(L.lib().aa_grpo_loss(lp.data_ptr(), lp.stride(0), ref_lp.data_ptr(), ref_lp.stride(0), L.dtype_code(lp.dtype),
                                     adv.data_ptr(), tokens.data_ptr(), tokens.stride(0), int(eos_id), B, K, float(beta),
                                     mode_code, loss.data_ptr(), grad.data_ptr(), grad.stride(0), row_end.data_ptr(),
                                     scratch.data_ptr(), sc['counter'][5:7].data_ptr(), L.stream_ptr(dev)))
        ctx.save_for_backward(grad)
        ctx.mark_non_differentiable(row_end)
        return loss[0], row_end

    @staticmethod
    def backward(ctx, g, _):
        (grad,) = ctx.saved_tensors
        return (grad.float() * g.float()).to(grad.dtype), None, None, None, None, None, None


def grpo_loss(per_token_logps: torch.Tensor, ref_per_token_logps: torch.Tensor, advantages: torch.Tensor,
              completion_tokens: torch.Tensor, eos_token_id: int, beta: float, mode: str | None = None):
    """The loss of GRPOTrainer.train_step (trainers/text_to_text/grpo.py:290-312): per-token k3 KL, per-token loss
    -(exp(lp - lp.detach()) * A - beta * KL), completion mask up to the first eos, token mean -> fp32 scalar,
    differentiable in per_token_logps.  Returns (loss, counted_tokens_per_row)."""
    L.require_cuda(per_token_logps, ref_per_token_logps, advantages, completion_tokens)
    if per_token_logps.dim() != 2 or per_token_logps.shape != ref_per_token_logps.shape or \
            completion_tokens.shape != per_token_logps.shape:
        raise ValueError('per-token log-probs and completion tokens must all be (B, K)')
    lp = _contiguous_last(per_token_logps)
    rlp = _contiguous_last(ref_per_token_logps.detach().to(lp.dtype))
    adv = advantages.detach().float().contiguous().view(-1)
    if adv.numel() != lp.size(0):
        raise ValueError('one advantage per sequence expected')
    tok = _contiguous_last(completion_tokens.to(torch.int64))
    return _GrpoLossFn.apply(lp, rlp, adv, tok, eos_token_id, beta, _mode_code(mode, lp.dtype))


def tail_token_log_probs(logits: torch.Tensor, input_ids: torch.Tensor, logits_to_keep: int, mode: str | None = None):
    """GRPOTrainer._get_per_token_logps after the model forward (trainers/text_to_text/grpo.py:205-210):
    log-probs of input_ids[:, -K:] under logits[:, :-1][:, -K:], one K1 launch, (B, K)."""
    L.require_cuda(logits, input_ids)
    B, seq, _ = logits.shape
    K = int(logits_to_keep)
    if not 0 < K < seq:
        raise ValueError('logits_to_keep must lie in (0, L)')
    logits = _contiguous_last(logits)
    lens = (K,) * B
    labels = strip_pad_tail(input_ids, lens, 0, strip=False)
    plan = _tail_plan(lens, seq, logits.stride(0), logits.stride(1), K, 0, -1, None, str(logits.device))
    return _LogProbFn.apply(logits, labels, plan, _mode_code(mode, logits.dtype))


class _GrpoFusedFn(torch.autograd.Function):
    """GRPO's policy log-probs, loss and d loss / d logits as ONE autograd node on K1f (aa_logprob_grpo_fused): the
    per-token loss needs the token's own log-prob, the reference log-prob and the sequence's advantage -- all there
    before the policy tile is read -- so the gradient tile is written in the same pass; aa_grpo_loss reduces the loss
    value from the log-probs that pass wrote."""

    @staticmethod
    def forward(ctx, logits, labels, plan, ref_lp, adv, tokens, eos_id, beta, mode_code):
        dev = logits.device
        B, K = plan.out_shape
        lp_dtype = logits.dtype if mode_code == L.MODE_FAITHFUL else torch.float32
        lp = torch.zeros((B, K), dtype=lp_dtype, device=dev)
        grad = torch.empty(logits.shape, dtype=logits.dtype, device=dev)
        rows = torch.empty(plan.n_tile_rows * 6, dtype=torch.int64, device=dev)  # 48 bytes per tile row
        row_end = torch.empty(B, dtype=torch.int32, device=dev)
        scratch = torch.empty(B + 1, dtype=torch.float32, device=dev)
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        sc = _device_scratch(dev)
        p = plan.ptrs()
        lib = L.lib()
        L.check(lib.aa_logprob_grpo_fused(
            logits.data_ptr(), L.dtype_code(logits.dtype), logits.stride(-2), logits.size(-1), labels.data_ptr(), plan.n_seg,
            p[0], p[1], p[2], p[3], p[4], plan.n_tile_rows, lp.data_ptr(), L.dtype_code(lp_dtype), ref_lp.data_ptr(),
            ref_lp.stride(0), adv.data_ptr(), tokens.data_ptr(), tokens.stride(0), int(eos_id), K, float(beta), mode_code,
            grad.data_ptr(), logits.size(-1), rows.data_ptr(), row_end.data_ptr(), scratch.data_ptr(),
            sc['counter'][5:6].data_ptr(), sc['status'].data_ptr(), L.stream_ptr(dev)))
        L.check(lib.aa_grpo_loss(lp.data_ptr(), lp.stride(0), ref_lp.data_ptr(), ref_lp.stride(0), L.dtype_code(lp_dtype),
                                 adv.data_ptr(), tokens.data_ptr(), tokens.stride(0), int(eos_id), B, K, float(beta),
                                 mode_code, loss.data_ptr(), None, 0, row_end.data_ptr(), scratch.data_ptr(),
                                 sc['counter'][5:7].data_ptr(), L.stream_ptr(dev)))
        ctx.save_for_backward(grad)
        ctx.consumed = False
        ctx.mark_non_differentiable(lp, row_end)
        return loss[0], lp, row_end

    @staticmethod
    def backward(ctx, g, _lp, _re):
        (grad,) = ctx.saved_tensors
        if ctx.consumed:
            raise RuntimeError('the single-pass GRPO node hands its gradient tile over once: set AA_B200_FUSED_GRPO=0 to '
                               'run backward twice through the same graph')
        ctx.consumed = True
        scale = g.detach().float().reshape(1).contiguous()
        L.check(L.lib().aa_scale_tile(grad.data_ptr(), L.dtype_code(grad.dtype), grad.numel(), scale.data_ptr(), L.AA_F32,
                                      L.stream_ptr(grad.device)))
        return grad, None, None, None, None, None, None, None, None


def grpo_loss_from_logits(logits: torch.Tensor, input_ids: torch.Tensor, logits_to_keep: int,
                          ref_per_token_logps: torch.Tensor, advantages: torch.Tensor, eos_token_id: int, beta: float,
                          mode: str | None = None):
    """`_get_per_token_logps` of the policy + the loss of GRPOTrainer.train_step (trainers/text_to_text/grpo.py:205-210,
    290-312) from the policy's logits; the reference model's per-token log-probs must already be there.
    -> (loss fp32 scalar, policy per-token log-probs (B, K), counted tokens per row).  With a gradient: one pass over the
    completion rows (see _GrpoFusedFn); otherwise tail_token_log_probs + grpo_loss."""
    L.require_cuda(logits, input_ids, ref_per_token_logps, advantages)
    K = int(logits_to_keep)
    tokens = input_ids[:, -K:]
    if not (_FUSED_GRPO and _single_pass_ok(logits) and torch.is_grad_enabled() and logits.requires_grad):
        lp = tail_token_log_probs(logits, input_ids, K, mode=mode)
        loss, row_end = grpo_loss(lp, ref_per_token_logps, advantages, tokens, eos_token_id, beta, mode=mode)
        return loss, lp.detach(), row_end
    B, seq, _ = logits.shape
    if not 0 < K < seq:
        raise ValueError('logits_to_keep must lie in (0, L)')
    if tuple(ref_per_token_logps.shape) != (B, K):
        raise ValueError('ref_per_token_logps must be (B, logits_to_keep)')
    logits = _contiguous_last(logits)
    mode_code = _mode_code(mode, logits.dtype)
    lp_dtype = logits.dtype if mode_code == L.MODE_FAITHFUL else torch.float32
    lens = (K,) * B
    labels = strip_pad_tail(input_ids, lens, 0, strip=False)
    plan = _tail_plan(lens, seq, logits.stride(0), logits.stride(1), K, 0, -1, None, str(logits.device))
    rlp = _contiguous_last(ref_per_token_logps.detach().to(lp_dtype))
    adv = advantages.detach().float().contiguous().view(-1)
    if adv.numel() != B:
        raise ValueError('one advantage per sequence expected')
    tok = _contiguous_last(tokens.to(torch.int64))
    return _GrpoFusedFn.apply(logits, labels, plan, rlp, adv, tok, int(eos_token_id), float(beta), mode_code)


# ---- reward-model pairwise loss -----------------------------------------------------------------------
class _RmPairLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, end_scores, regularization):
        n = end_scores.numel()
        dev = end_scores.device
        out = torch.empty(2, dtype=torch.float32, device=dev)
        grad = torch.empty(n, dtype=torch.float32, device=dev)
        L.check(L.lib().aa_rm_pair_loss(end_scores.data_ptr(), n // 2, float(regularization), out.data_ptr(),
                                        grad.data_ptr(), L.stream_ptr(dev)))
        ctx.save_for_backward(grad)
        ctx.shape = end_scores.shape
        ctx.mark_non_differentiable(out)
        return out[0].clone(), out

    @staticmethod
    def backward(ctx, g, _):
        (grad,) = ctx.saved_tensors
        return (grad * g).view(ctx.shape), None


def rm_pair_loss(end_scores: torch.Tensor, regularization: float = 0.0) -> dict[str, torch.Tensor]:
    """The loss tail of RMTrainer.loss (trainers/text_to_text/rm.py:111-124): end_scores (2B,) or (2B, 1)
    fp32, higher rows first -> {'loss', 'accuracy', 'higher_end_reward', 'lower_end_reward'}; one launch for
    forward + backward."""
    L.require_cuda(end_scores)
    flat = end_scores.reshape(-1)
    if flat.numel() % 2:
        raise ValueError('end_scores must hold 2B values (higher first, lower second)')
    flat = flat.float().contiguous()
    loss, out = _RmPairLossFn.apply(flat, regularization)
    higher, lower = flat.detach().chunk(2)
    return {'loss': loss, 'accuracy': out[1], 'higher_end_reward': higher, 'lower_end_reward': lower, '_stats': out}


# ---- causal-LM cross-entropy (SFT loss, PPO ptx term) -------------------------------------------------
class _CausalLMLossFn(torch.autograd.Function):
    """Mean NLL over labels != ignore_index, times `loss_scale`.
    With a gradient (default, K1f): ONE pass over the valid rows produces the fp32 log-probs AND the gradient tile
    (every valid row's upstream gradient is the same -loss_scale / n_valid, counted on the device before the pass;
    each row is streamed twice by one CTA, the second time out of L2); backward hands the tile over, multiplied in
    place only if the incoming scalar is not 1.  AA_B200_FUSED_CE=0 / no gradient: K1 in fp32 mode over every
    position (ignored labels cost no traffic), mean-NLL epilogue; backward: one K1b launch with the scalar
    -loss_scale / n_valid as upstream gradient.  -> (loss_scale * loss, loss)."""

    @staticmethod
    def forward(ctx, logits, shift_labels, ignore_index, loss_scale):
        B, seq, V = logits.shape
        dev = logits.device
        plan = _dense_plan(B, seq, logits.stride(0) if B > 1 else seq * logits.stride(1), logits.stride(1), seq, 0, seq,
                           B * seq, str(dev))
        need_grad = ctx.needs_input_grad[0]
        ctx.fused = bool(_FUSED_CE and need_grad and _single_pass_ok(logits))
        sc = _device_scratch(dev)
        out = torch.empty(3, dtype=torch.float32, device=dev)  # [loss, -1 / n_valid, -loss_scale / n_valid]
        if ctx.fused:
            logp = torch.zeros((B, seq), dtype=torch.float32, device=dev)
            grad = torch.empty(logits.shape, dtype=logits.dtype, device=dev)
            scratch = torch.empty(B * seq * 6, dtype=torch.int64, device=dev)  # 48 bytes per tile row
            p = plan.ptrs()
            L.check(L.lib().aa_logprob_ce_fused(
                logits.data_ptr(), L.dtype_code(logits.dtype), logits.stride(-2), V, shift_labels.data_ptr(), B * seq,
                int(ignore_index), plan.n_seg, p[0], p[1], p[2], p[3], p[4], B * seq, logp.data_ptr(), float(loss_scale),
                grad.data_ptr(), V, scratch.data_ptr(), out[2:3].data_ptr(), sc['status'].data_ptr(), L.stream_ptr(dev)))
        else:
            logp = torch.empty((B, seq), dtype=torch.float32, device=dev)
            stats = torch.empty((2, B * seq), dtype=torch.float32, device=dev) if need_grad else None
            _launch_fwd(logits, shift_labels, plan, logp, stats[0] if need_grad else None, stats[1] if need_grad else None,
                        ignore_index=ignore_index)
        partial = torch.empty(512, dtype=torch.float32, device=dev)
        L.check(L.lib().aa_nll_mean(logp.data_ptr(), L.AA_F32, shift_labels.data_ptr(), B * seq, int(ignore_index),
                                    out[0:1].data_ptr(), out[1:2].data_ptr(), partial.data_ptr(),
                                    sc['counter'][4:5].data_ptr(), L.stream_ptr(dev)))
        if ctx.fused:
            ctx.save_for_backward(grad)
            ctx.consumed = False
        elif need_grad:
            ctx.save_for_backward(logits, shift_labels, stats, out)
            ctx.plan, ctx.ignore_index = plan, int(ignore_index)
        ctx.loss_scale = float(loss_scale)
        loss = out[0]
        scaled = loss if loss_scale == 1.0 else loss * float(loss_scale)
        ctx.mark_non_differentiable(loss)
        return scaled.clone() if scaled is loss else scaled, loss

    @staticmethod
    def backward(ctx, g, _unused):
        if ctx.fused:
            (grad,) = ctx.saved_tensors
            if ctx.consumed:
                raise RuntimeError('the single-pass cross-entropy node hands its gradient tile over once: set '
                                   'AA_B200_FUSED_CE=0 to run backward twice through the same graph')
            ctx.consumed = True
            scale = g.detach().float().reshape(1).contiguous()
            L.check(L.lib().aa_scale_tile(grad.data_ptr(), L.dtype_code(grad.dtype), grad.numel(), scale.data_ptr(),
                                          L.AA_F32, L.stream_ptr(grad.device)))
            return grad, None, None, None
        logits, shift_labels, stats, out = ctx.saved_tensors
        grad = torch.empty(logits.shape, dtype=logits.dtype, device=logits.device)
        scale = (out[1] * (g.float() * ctx.loss_scale)).reshape(1).contiguous()
        _launch_bwd(logits, shift_labels, ctx.plan, stats[0], stats[1], None, None, scale, grad, L.MODE_F32,
                    ignore_index=ctx.ignore_index)
        return grad, None, None, None


def _shifted_labels(logits: torch.Tensor, labels: torch.Tensor, ignore_index: int):
    L.require_cuda(logits, labels)
    if logits.dim() != 3 or labels.shape != logits.shape[:2]:
        raise ValueError('expected logits (B, L, V) and labels (B, L)')
    logits = _contiguous_last(logits)
    if logits.size(0) > 1 and logits.stride(0) != logits.size(1) * logits.stride(1):
        logits = logits.contiguous()
    shift = torch.full(labels.shape, int(ignore_index), dtype=torch.int64, device=labels.device)
    shift[:, :-1] = labels[:, 1:]
    return logits, shift


def causal_lm_loss(logits: torch.Tensor, labels: torch.Tensor, ignore_index: int = -100) -> torch.Tensor:
    """The `outputs.loss` of an HF causal LM (transformers ForCausalLMLoss: logits upcast to fp32, labels
    shifted by one, mean cross-entropy over labels != ignore_index) without the fp32 copy of the logits
    tile or the (rows, V) log-softmax tile: the loss of SupervisedTrainer.loss
    (trainers/text_to_text/sft.py:95-98) and of PPOTrainer.ptx_step (trainers/text_to_text/ppo.py:400-408).
    logits (B, L, V) in the model dtype, labels (B, L) -> fp32 scalar, differentiable in logits."""
    logits, shift = _shifted_labels(logits, labels, ignore_index)
    return _CausalLMLossFn.apply(logits, shift, int(ignore_index), 1.0)[0]


def causal_lm_loss_scaled(logits: torch.Tensor, labels: torch.Tensor, loss_scale: float, ignore_index: int = -100):
    """-> (loss_scale * loss, loss.detach()).  Backpropagate the FIRST: the gradient tile is born multiplied by
    `loss_scale` (ptx_step's `ptx_coeff * ptx_loss`, trainers/text_to_text/ppo.py:405), so no pass over the tile is spent
    on the multiplication; log the second."""
    logits, shift = _shifted_labels(logits, labels, ignore_index)
    return _CausalLMLossFn.apply(logits, shift, int(ignore_index), float(loss_scale))



# ---- the same cross-entropy from the last hidden states (fused lm_head: no logits tile) -------------------------
class CERows:
    """The rows a causal-LM cross-entropy scores, compacted on the device by ONE aa_ce_rows launch: flat indices
    b * L + t of the positions whose shifted label labels[b, t + 1] != ignore_index, in ascending order, and those labels.

    The lm_head kernels are sized by the number of valid rows, which only the device knows.  The count is copied into
    pinned host memory right after the launch and an event is recorded behind the copy; n_valid() waits on that event.
    The trainers build the plan BEFORE they enqueue the model forward (the stream is idle then: the previous step ended
    with its host read) and read n_valid() AFTER it, so by the time the host asks, the copy finished long ago and neither
    the host nor the device waits on the other."""

    __slots__ = ('shape', 'vocab_size', 'ignore_index', '_index', '_labels', '_count', '_host', '_event', '_n')

    def __init__(self, labels: torch.Tensor, vocab_size: int, ignore_index: int):
        L.require_cuda(labels)
        if labels.dim() != 2:
            raise ValueError(f'expected labels (B, L), got {tuple(labels.shape)}')
        if labels.dtype != torch.int64:
            labels = labels.to(torch.int64)
        B, seq = labels.shape
        self.shape, self.vocab_size, self.ignore_index = (B, seq), int(vocab_size), int(ignore_index)
        dev = labels.device
        self._index = torch.empty(B * seq, dtype=torch.int64, device=dev)
        self._labels = torch.empty(B * seq, dtype=torch.int64, device=dev)
        self._count = torch.zeros(1, dtype=torch.int64, device=dev)
        self._host = self._event = self._n = None
        if B * seq == 0:
            self._n = 0
            return
        L.check(L.lib().aa_ce_rows(labels.data_ptr(), B, seq, labels.stride(0), labels.stride(1), self.ignore_index,
                                   self.vocab_size, self._index.data_ptr(), self._labels.data_ptr(), self._count.data_ptr(),
                                   _device_scratch(dev)['status'].data_ptr(), L.stream_ptr(dev)))
        self._start_count_copy()

    def _start_count_copy(self):
        self._host = torch.empty(1, dtype=torch.int64, pin_memory=True)
        self._host.copy_(self._count, non_blocking=True)
        self._event = torch.cuda.Event()
        self._event.record(torch.cuda.current_stream(self._count.device))

    def n_valid(self) -> int:
        """The number of valid rows (host int): waits on the count copy, once."""
        if self._n is None:
            self._event.synchronize()
            self._n = int(self._host[0])
        return self._n

    @property
    def index(self) -> torch.Tensor:
        return self._index[:self.n_valid()]

    @property
    def labels(self) -> torch.Tensor:
        return self._labels[:self.n_valid()]


def ce_rows(labels: torch.Tensor, vocab_size: int, ignore_index: int = -100) -> CERows:
    """The row plan of causal_lm_loss_from_hidden for labels (B, L): one launch, an asynchronous copy of the count, no host
    wait.  Call it before the model forward is enqueued (see CERows).  A label outside [0, vocab_size) other than
    ignore_index sets the device status word (raise_for_status raises IndexError, as ATen's cross_entropy would)."""
    return CERows(labels, vocab_size, ignore_index)


class _MeanNllFn(torch.autograd.Function):
    """loss_scale * mean(-lp) over the compact rows: ONE aa_nll_mean launch -> (loss_scale * loss, loss).  Backward: the
    per-row upstream gradient -loss_scale * g / n_valid, which the lm_head node folds into its d(logits) pass."""

    @staticmethod
    def forward(ctx, lp, labels, ignore_index, loss_scale):
        dev = lp.device
        sc = _device_scratch(dev)
        out = torch.empty(2, dtype=torch.float32, device=dev)  # [loss, -1 / n_valid]
        partial = torch.empty(512, dtype=torch.float32, device=dev)
        L.check(L.lib().aa_nll_mean(lp.data_ptr(), L.AA_F32, labels.data_ptr(), lp.numel(), int(ignore_index),
                                    out[0:1].data_ptr(), out[1:2].data_ptr(), partial.data_ptr(),
                                    sc['counter'][4:5].data_ptr(), L.stream_ptr(dev)))
        ctx.save_for_backward(out)
        ctx.n, ctx.loss_scale = lp.numel(), float(loss_scale)
        loss = out[0]
        scaled = loss if loss_scale == 1.0 else loss * float(loss_scale)
        ctx.mark_non_differentiable(loss)
        return scaled.clone() if scaled is loss else scaled, loss

    @staticmethod
    def backward(ctx, g, _unused):
        (out,) = ctx.saved_tensors
        return (out[1] * (g.float() * ctx.loss_scale)).expand(ctx.n), None, None, None


class _NoValidRowsFn(torch.autograd.Function):
    """Every label ignored: the loss is NaN (causal_lm_loss's 0 / 0), the gradients are zero, no lm_head work."""

    @staticmethod
    def forward(ctx, hidden, weight, loss_scale):
        ctx.meta = (hidden.shape, hidden.dtype, weight.shape, weight.dtype, hidden.device)
        loss = torch.full((), float('nan'), dtype=torch.float32, device=hidden.device)
        ctx.mark_non_differentiable(loss)
        return loss.clone(), loss

    @staticmethod
    def backward(ctx, g, _unused):
        hs, hd, ws, wd, dev = ctx.meta
        dh = torch.zeros(hs, dtype=hd, device=dev) if ctx.needs_input_grad[0] else None
        dw = torch.zeros(ws, dtype=wd, device=dev) if ctx.needs_input_grad[1] else None
        return dh, dw, None


def causal_lm_loss_from_hidden_scaled(hidden: torch.Tensor, weight: torch.Tensor, labels: torch.Tensor, loss_scale: float,
                                      ignore_index: int = -100, chunk_rows: int | None = None, rows: CERows | None = None):
    """causal_lm_loss_scaled(F.linear(hidden, weight), labels, loss_scale) without the (B, L, V) logits tile or its
    gradient -> (loss_scale * loss, loss.detach()).  hidden (B, L, H) = the model's last hidden states, weight (V, H) = its
    bias-free lm_head (lm_head_weight), labels (B, L).  Only the valid rows are gathered (rows: the ce_rows plan, built
    here if not given) into a compact (n_valid, H) matrix for linear_token_log_probs in the cross-entropy's rounding
    (bf16 operands, H % 64 == 0: K6 forward, K6b + the two tcgen05 GEMMs backward; otherwise chunked library GEMMs around
    K1 / K1b); the mean is one aa_nll_mean launch.  Differentiable in hidden and weight."""
    L.require_cuda(hidden, weight, labels)
    if hidden.dim() != 3 or weight.dim() != 2 or hidden.size(2) != weight.size(1) or labels.shape != hidden.shape[:2]:
        raise ValueError(f'expected hidden (B, L, H), weight (V, H), labels (B, L); got {tuple(hidden.shape)}, '
                         f'{tuple(weight.shape)}, {tuple(labels.shape)}')
    if rows is None:
        rows = ce_rows(labels, weight.size(0), ignore_index)
    elif rows.shape != tuple(labels.shape) or rows.ignore_index != int(ignore_index) or rows.vocab_size != weight.size(0):
        raise ValueError('the CERows plan was built for other labels, ignore_index or vocabulary')
    n = rows.n_valid()  # the one host wait of this path; see CERows
    if n == 0:
        return _NoValidRowsFn.apply(hidden, weight, float(loss_scale))
    B, seq, H = hidden.shape
    labels_c = rows.labels
    x = hidden.reshape(B * seq, H).index_select(0, rows.index)
    lp = linear_token_log_probs(x, weight, labels_c, chunk_rows, mode='ce')
    return _MeanNllFn.apply(lp, labels_c, int(ignore_index), float(loss_scale))


def causal_lm_loss_from_hidden(hidden: torch.Tensor, weight: torch.Tensor, labels: torch.Tensor, ignore_index: int = -100,
                               chunk_rows: int | None = None, rows: CERows | None = None) -> torch.Tensor:
    """causal_lm_loss(F.linear(hidden, weight), labels) without the logits tile: fp32 scalar, differentiable in hidden
    and weight (see causal_lm_loss_from_hidden_scaled)."""
    return causal_lm_loss_from_hidden_scaled(hidden, weight, labels, 1.0, ignore_index, chunk_rows, rows)[0]


# ---- masked mean ---------------------------------------------------------------------------------
class _MaskedMeanFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, m):
        B, W = x.shape
        dev = x.device
        out = torch.empty(1, dtype=torch.float32, device=dev)
        rows = torch.empty(B, dtype=torch.float32, device=dev)
        sc = _device_scratch(dev)
        L.check(L.lib().aa_masked_mean(x.data_ptr(), L.dtype_code(x.dtype), x.stride(0), L.ptr(m),
                                       m.stride(0) if m is not None else 0, B, W, out.data_ptr(), rows.data_ptr(),
                                       sc['counter'][1:2].data_ptr(), L.stream_ptr(dev)))
        ctx.save_for_backward(m)
        ctx.shape, ctx.dtype = x.shape, x.dtype
        return out[0]

    @staticmethod
    def backward(ctx, g):
        (m,) = ctx.saved_tensors
        B, W = ctx.shape
        if m is None:
            return (g / (B * W)).to(ctx.dtype).expand(B, W), None
        coef = g / (B * m.sum(dim=-1, keepdim=True).float())
        return (m * coef).to(ctx.dtype), None


def masked_mean(x: torch.Tensor, mask: torch.Tensor | None = None) -> torch.Tensor:
    """utils/tools.py:460-467: mean over rows of masked row means -> fp32 scalar (NaN when a row is
    fully masked, like the reference).  Differentiable in x."""
    L.require_cuda(x, mask)
    if x.dim() != 2:
        raise ValueError('masked_mean expects (B, L)')
    x = _contiguous_last(x)
    if x.dtype not in (torch.float32, torch.bfloat16, torch.float16):
        x = x.float()
    m = None
    if mask is not None:
        m = _contiguous_last(mask.to(torch.bool))
    return _MaskedMeanFn.apply(x, m)


# ---- K3 score head -------------------------------------------------------------------------------
class _ScoreHeadFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, hidden, weight, out_dtype, mode_code):
        Bsz, seq, H = hidden.shape
        dev = hidden.device
        scores = torch.empty((Bsz, seq), dtype=out_dtype, device=dev)
        L.check(L.lib().aa_score_head_fwd(hidden.data_ptr(), L.dtype_code(hidden.dtype), Bsz * seq, H,
                                          hidden.stride(1), weight.data_ptr(), scores.data_ptr(),
                                          L.dtype_code(out_dtype), mode_code, L.stream_ptr(dev)))
        ctx.save_for_backward(hidden, weight)
        ctx.mode_code = mode_code
        return scores

    @staticmethod
    def backward(ctx, g):
        hidden, weight = ctx.saved_tensors
        Bsz, seq, H = hidden.shape
        dev = hidden.device
        g = g.contiguous()
        if g.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            g = g.float()
        if ctx.mode_code == L.MODE_FAITHFUL and g.dtype != hidden.dtype:
            # `.float()` after nn.Linear: autograd casts the incoming gradient back to the hidden dtype first
            g = g.to(hidden.dtype)
        need_h, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        grad_hidden = torch.empty_like(hidden, memory_format=torch.contiguous_format) if need_h else None
        grad_w32 = torch.empty(H, dtype=torch.float32, device=dev)
        import ctypes

        n_part = ctypes.c_int32(0)
        lib = L.lib()
        common = (hidden.data_ptr(), L.dtype_code(hidden.dtype), Bsz * seq, H, hidden.stride(1), weight.data_ptr(),
                  g.data_ptr(), L.dtype_code(g.dtype), L.ptr(grad_hidden), H, grad_w32.data_ptr())
        L.check(lib.aa_score_head_bwd(*common, None, ctypes.byref(n_part), ctx.mode_code, L.stream_ptr(dev)))
        partial = torch.empty((n_part.value, H), dtype=torch.float32, device=dev)
        L.check(lib.aa_score_head_bwd(*common, partial.data_ptr(), ctypes.byref(n_part), ctx.mode_code,
                                      L.stream_ptr(dev)))
        grad_w = grad_w32.to(weight.dtype).view_as(weight) if need_w else None
        return grad_hidden, grad_w, None, None


def score_head(last_hidden: torch.Tensor, weight: torch.Tensor, upcast: bool = True, mode: str | None = None):
    """scores = score_head(last_hidden_state)[.float()]  (models/llama.py:62-63; qwen2_vl.py:59-60 keeps
    the hidden dtype: upcast=False).  last_hidden (B, L, H), weight (1, H) or (H,) -> (B, L)."""
    L.require_cuda(last_hidden, weight)
    if last_hidden.dim() != 3:
        raise ValueError('last_hidden must be (B, L, H)')
    H = last_hidden.size(-1)
    if weight.numel() != H:
        raise ValueError('score_head weight must have H elements (nn.Linear(H, 1, bias=False))')
    hidden = last_hidden
    if hidden.stride(-1) != 1 or hidden.stride(0) != hidden.size(1) * hidden.stride(1) or \
            (hidden.stride(1) * hidden.element_size()) % 16 or hidden.data_ptr() % 16:
        hidden = hidden.contiguous()
    w = weight.to(hidden.dtype).contiguous()
    mode_code = _mode_code(mode, hidden.dtype)
    out_dtype = torch.float32 if (upcast or mode_code == L.MODE_F32) else hidden.dtype
    return _ScoreHeadFn.apply(hidden, w, out_dtype, mode_code)


def score_end(scores: torch.Tensor, attention_mask: torch.Tensor | None, last_hidden: torch.Tensor | None = None):
    """end_index / end_scores / end_last_hidden_state (models/llama.py:71-93): last attended position
    per row (attention_mask given) or position L-1 (attention_mask None: llava.py:64-66,
    qwen2_vl.py:62-64).  No host sync (the reference loops `m.nonzero()[-1]` per sample)."""
    L.require_cuda(scores, attention_mask, last_hidden)
    B, seq = scores.shape
    dev = scores.device
    scores = _contiguous_last(scores.detach())
    mask = None
    kind = L.MASK_U8
    if attention_mask is not None:
        mask = attention_mask
        if mask.dtype == torch.bool:
            mask = _contiguous_last(mask)
        elif mask.dtype == torch.int64:
            kind = L.MASK_I64
            mask = _contiguous_last(mask)
        else:
            mask = _contiguous_last(mask != 0)
    end_index = torch.empty(B, dtype=torch.int64, device=dev)
    end_scores = torch.empty(B, dtype=torch.float32, device=dev)
    end_hidden = None
    hid = None
    if last_hidden is not None:
        hid = _contiguous_last(last_hidden.detach())
        end_hidden = torch.empty((B, hid.size(-1)), dtype=hid.dtype, device=dev)
    sc = _device_scratch(dev)
    L.check(L.lib().aa_score_end(
        scores.data_ptr(), L.dtype_code(scores.dtype), scores.stride(0), L.ptr(mask), kind,
        mask.stride(0) if mask is not None else 0, B, seq, end_index.data_ptr(), end_scores.data_ptr(),
        L.ptr(hid), L.dtype_code(hid.dtype) if hid is not None else L.AA_F32,
        hid.stride(0) if hid is not None else 0, hid.stride(1) if hid is not None else 0,
        hid.size(-1) if hid is not None else 0, L.ptr(end_hidden), sc['status'].data_ptr(), L.stream_ptr(dev)))
    return end_index, end_scores, end_hidden


# ---- K4 / K5 PPO ---------------------------------------------------------------------------------
def _promote(a: torch.dtype, b: torch.dtype) -> torch.dtype:
    return a if a == b else torch.float32


def kl_rewards_and_gae(reward, log_probs, ref_log_probs, values, sequence_mask, start: int, kl_coeff: float,
                       clip_range_score: float, gamma: float, gae_lambda: float, mode: str | None = None):
    """add_kl_divergence_regularization (trainers/text_to_text/ppo.py:528-547) +
    get_advantages_and_returns (:487-508) in ONE launch (K4).  Returns
    (old_rewards (B, W), advantages (B, W-start), returns (B, W-start), row_stats (B, 8) fp32)."""
    L.require_cuda(reward, log_probs, ref_log_probs, values, sequence_mask)
    if log_probs.dim() != 2:
        raise ValueError('log_probs must be (B, W)')
    B, W = log_probs.shape
    # the kernel indexes every (B, W) operand with W taken from log_probs: a narrower mask / values tensor would be
    # read past its end (the reference's elementwise ops raise a broadcast error instead)
    if not (tuple(ref_log_probs.shape) == tuple(values.shape) == tuple(sequence_mask.shape) == (B, W)):
        raise ValueError(f'ref_log_probs {tuple(ref_log_probs.shape)}, values {tuple(values.shape)} and sequence_mask '
                         f'{tuple(sequence_mask.shape)} must all match log_probs {(B, W)}')
    if reward.numel() != B:
        raise ValueError(f'reward must hold one value per sample ({B}); got {tuple(reward.shape)}')
    dev = log_probs.device
    lp = _contiguous_last(log_probs.detach())
    rlp = ref_log_probs.detach().to(lp.dtype)
    rlp = rlp if rlp.stride() == lp.stride() else rlp.contiguous()
    if rlp.stride() != lp.stride():
        lp = lp.contiguous()
    vals = _contiguous_last(values.detach())
    mask = _contiguous_last(sequence_mask.to(torch.bool))
    rew = reward.detach().to(torch.float32).contiguous()
    mode_code = _mode_code(mode, lp.dtype)
    faithful = mode_code == L.MODE_FAITHFUL
    rew_dtype = lp.dtype if faithful else torch.float32
    adv_dtype = _promote(vals.dtype, lp.dtype) if faithful else torch.float32
    old_rewards = torch.empty((B, W), dtype=rew_dtype, device=dev)
    adv = torch.empty((B, W - start), dtype=adv_dtype, device=dev)
    ret = torch.empty((B, W - start), dtype=adv_dtype, device=dev)
    row_stats = torch.empty((B, 8), dtype=torch.float32, device=dev)
    sc = _device_scratch(dev)
    L.check(L.lib().aa_ppo_prep(
        lp.data_ptr(), rlp.data_ptr(), L.dtype_code(lp.dtype), lp.stride(0), rew.data_ptr(), vals.data_ptr(),
        L.dtype_code(vals.dtype), vals.stride(0), mask.data_ptr(), mask.stride(0), B, W, int(start),
        float(kl_coeff), float(clip_range_score), float(gamma), float(gae_lambda), mode_code,
        old_rewards.data_ptr(), L.dtype_code(rew_dtype), adv.data_ptr(), ret.data_ptr(), L.dtype_code(adv_dtype),
        row_stats.data_ptr(), sc['status'].data_ptr(), L.stream_ptr(dev)))
    return old_rewards, adv, ret, row_stats


def gae_from_rewards(values, rewards, sequence_mask, start: int, gamma: float, gae_lambda: float,
                     mode: str | None = None):
    """PPOTrainer.get_advantages_and_returns on its own (trainers/text_to_text/ppo.py:487-508): the
    GAE half of K4 on precomputed per-token rewards.  Returns (advantages, returns, row_stats)."""
    L.require_cuda(values, rewards, sequence_mask)
    if rewards.dim() != 2 or not (tuple(values.shape) == tuple(sequence_mask.shape) == tuple(rewards.shape)):
        raise ValueError(f'values {tuple(values.shape)}, rewards {tuple(rewards.shape)} and sequence_mask '
                         f'{tuple(sequence_mask.shape)} must share one (B, W) shape')
    B, W = rewards.shape
    dev = rewards.device
    rew = rewards.detach().contiguous()
    if rew.dtype not in (torch.float32, torch.bfloat16, torch.float16):
        rew = rew.float()
    vals = _contiguous_last(values.detach())
    mask = _contiguous_last(sequence_mask.to(torch.bool))
    mode_code = _mode_code(mode, rew.dtype)
    faithful = mode_code == L.MODE_FAITHFUL
    adv_dtype = _promote(vals.dtype, rew.dtype) if faithful else torch.float32
    adv = torch.empty((B, W - start), dtype=adv_dtype, device=dev)
    ret = torch.empty((B, W - start), dtype=adv_dtype, device=dev)
    row_stats = torch.empty((B, 8), dtype=torch.float32, device=dev)
    sc = _device_scratch(dev)
    L.check(L.lib().aa_ppo_prep(
        None, None, L.dtype_code(rew.dtype), 0, None, vals.data_ptr(), L.dtype_code(vals.dtype), vals.stride(0),
        mask.data_ptr(), mask.stride(0), B, W, int(start), 0.0, 0.0, float(gamma), float(gae_lambda), mode_code,
        rew.data_ptr(), L.dtype_code(rew.dtype), adv.data_ptr(), ret.data_ptr(), L.dtype_code(adv_dtype),
        row_stats.data_ptr(), sc['status'].data_ptr(), L.stream_ptr(dev)))
    return adv, ret, row_stats


def _ppo_loss_launch(x, old, aux, mask, clip, mode_code, actor: bool, x_tail=None):
    """K5: -> (loss fp32[2], loss as a 0-dim tensor of the promoted dtype (a view, no launch), grad (B, Wm), row_mean).
    x_tail = (DeviceLens, src_width): `x` is the raw (B, src_width) tensor and the kernel reads the per-sample tails."""
    B, Wm = old.shape
    dev = x.device
    loss = torch.empty(2, dtype=torch.float32, device=dev)
    grad = torch.empty((B, Wm), dtype=x.dtype, device=dev)
    rows = torch.empty(B, dtype=torch.float32, device=dev)
    row_mean = torch.empty(B, dtype=torch.float32, device=dev)
    sc = _device_scratch(dev)
    lib = L.lib()
    if actor:
        L.check(lib.aa_ppo_actor_loss(
            x.data_ptr(), x.stride(0), old.data_ptr(), old.stride(0), L.dtype_code(x.dtype), aux.data_ptr(),
            aux.stride(0), L.dtype_code(aux.dtype), mask.data_ptr(), mask.stride(0), B, Wm, float(clip),
            mode_code, loss.data_ptr(), grad.data_ptr(), grad.stride(0), rows.data_ptr(),
            sc['counter'][2:3].data_ptr(), L.stream_ptr(dev)))
    else:
        L.check(lib.aa_ppo_critic_loss(
            x.data_ptr(), x.stride(0), old.data_ptr(), old.stride(0), L.dtype_code(x.dtype), aux.data_ptr(),
            aux.stride(0), L.dtype_code(aux.dtype), mask.data_ptr(), mask.stride(0), B, Wm, float(clip),
            mode_code, loss.data_ptr(), grad.data_ptr(), grad.stride(0), row_mean.data_ptr(), rows.data_ptr(),
            sc['counter'][3:4].data_ptr(), x_tail[0].dev.data_ptr() if x_tail else None, int(x_tail[1]) if x_tail else 0,
            L.stream_ptr(dev)))
    out_dtype = _promote(x.dtype, aux.dtype) if mode_code == L.MODE_FAITHFUL else torch.float32
    cast = loss[0] if out_dtype == torch.float32 else loss[1:2].view(out_dtype)[0]
    return loss, cast, grad, row_mean


class _PpoLossFn(torch.autograd.Function):
    """K5: forward computes the loss AND d loss / d x in the same launch; backward scales it."""

    @staticmethod
    def forward(ctx, x, old, aux, mask, clip, mode_code, actor: bool):
        loss, cast, grad, row_mean = _ppo_loss_launch(x, old, aux, mask, clip, mode_code, actor)
        ctx.save_for_backward(grad)
        ctx.mark_non_differentiable(row_mean, loss)
        return cast, row_mean, loss

    @staticmethod
    def backward(ctx, g_loss, _g, _l):
        (grad,) = ctx.saved_tensors
        return (grad.float() * g_loss.float()).to(grad.dtype), None, None, None, None, None, None


class _TailActorLossFn(torch.autograd.Function):
    """The actor half of the multimodal rl_step as ONE autograd node (trainers/text_image_to_text/ppo.py:298-316).

    Default (K1f, aa_logprob_actor_fused): the forward makes ONE pass over the scored rows and already writes the
    gradient tile -- the objective is a masked mean of per-token terms, so d loss / d log-prob needs nothing but the
    token's own log-prob; each row is streamed twice by the same CTA and the second pass comes out of L2.  K5 then reduces
    the loss value from the log-probs; backward hands the tile over (aa_scale_tile multiplies it by the incoming scalar
    on the device iff that is not 1).
    AA_B200_FUSED_ACTOR=0 (and rows without gradient): forward = K1 over the response tails + K5; backward = K1b taking
    K5's d loss / d log-probs as its per-row upstream gradient and the incoming scalar as a device scale."""

    @staticmethod
    def forward(ctx, logits, ids, plan, old, aux, mask, clip, mode_code):
        out_dtype = logits.dtype if mode_code == L.MODE_FAITHFUL else torch.float32
        dev = logits.device
        lp = torch.zeros(plan.out_shape, dtype=out_dtype, device=dev)
        ctx.fused = bool(_FUSED_ACTOR and _single_pass_ok(logits) and ctx.needs_input_grad[0] and plan.n_tile_rows > 0 and plan.n_seg > 0
                         and plan.n_tile_rows % plan.n_seg == 0 and len(plan.out_shape) == 2)
        if ctx.fused:
            grad = torch.empty(logits.shape, dtype=logits.dtype, device=dev)
            scratch = torch.empty(plan.n_tile_rows * 6, dtype=torch.int64, device=dev)  # 48 bytes per tile row
            p = plan.ptrs()
            L.check(L.lib().aa_logprob_actor_fused(
                logits.data_ptr(), L.dtype_code(logits.dtype), logits.stride(-2), logits.size(-1), ids.data_ptr(),
                plan.n_seg, p[0], p[1], p[2], p[3], p[4], plan.n_tile_rows, lp.data_ptr(), L.dtype_code(lp.dtype),
                None, None, old.data_ptr(), old.stride(0), aux.data_ptr(), aux.stride(0), L.dtype_code(aux.dtype),
                mask.data_ptr(), mask.stride(0), lp.size(1), float(clip), mode_code, grad.data_ptr(), logits.size(-1),
                scratch.data_ptr(), _device_scratch(dev)['status'].data_ptr(), L.stream_ptr(dev)))
            loss, cast, _, _ = _ppo_loss_launch(lp, old, aux, mask, clip, mode_code, True)
            ctx.save_for_backward(grad)
            ctx.consumed = False
        else:
            stats = torch.empty((2, max(plan.n_rows, 1)), dtype=torch.float32, device=dev)
            _launch_fwd(logits, ids, plan, lp, stats[0], stats[1])
            loss, cast, grad, _ = _ppo_loss_launch(lp, old, aux, mask, clip, mode_code, True)
            ctx.save_for_backward(logits, ids, stats, grad)
            ctx.plan, ctx.mode_code = plan, mode_code
        ctx.mark_non_differentiable(lp, loss)
        return cast, lp, loss

    @staticmethod
    def backward(ctx, g_loss, _lp, _l):
        scale = g_loss.detach().reshape(1)
        if scale.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            scale = scale.float()
        scale = scale.contiguous()
        if ctx.fused:
            (grad,) = ctx.saved_tensors
            if ctx.consumed:
                raise RuntimeError('the single-pass actor node hands its gradient tile over once: set '
                                   'AA_B200_FUSED_ACTOR=0 to run backward twice through the same graph')
            ctx.consumed = True
            L.check(L.lib().aa_scale_tile(grad.data_ptr(), L.dtype_code(grad.dtype), grad.numel(), scale.data_ptr(),
                                          L.dtype_code(scale.dtype), L.stream_ptr(grad.device)))
            return grad, None, None, None, None, None, None, None
        logits, ids, stats, grad_lp = ctx.saved_tensors
        grad = torch.empty(logits.shape, dtype=logits.dtype, device=logits.device)
        _launch_bwd(logits, ids, ctx.plan, stats[0], stats[1], grad_lp, None, scale, grad, ctx.mode_code)
        return grad, None, None, None, None, None, None, None


class _TailCriticLossFn(torch.autograd.Function):
    """The critic half (text_image_to_text/ppo.py:318-337): forward = K5 reading `scores.squeeze(-1)[:, :-1]` through
    the per-sample tail indexing; backward = ONE launch that scatters K5's gradient back into the raw (B, L[, 1]) scores
    layout, zeros and the upstream scalar included."""

    @staticmethod
    def forward(ctx, scores, lens_dev, bound, old, aux, mask, clip, mode_code):
        raw = scores.squeeze(-1) if scores.dim() == 3 else scores  # (B, L)
        raw = _contiguous_last(raw)
        src_width = raw.size(1) - 1  # `[:, :-1]`
        lens = DeviceLens(lens_dev, bound)
        loss, cast, grad, row_mean = _ppo_loss_launch(raw, old, aux, mask, clip, mode_code, False, x_tail=(lens, src_width))
        ctx.save_for_backward(grad, lens_dev)
        ctx.shape, ctx.src_width = scores.shape, src_width
        ctx.mark_non_differentiable(row_mean, loss)
        return cast, row_mean, loss

    @staticmethod
    def backward(ctx, g_loss, _r, _l):
        grad, lens_dev = ctx.saved_tensors
        B, W = grad.shape
        Lq = ctx.src_width + 1
        out = torch.empty((B, Lq), dtype=grad.dtype, device=grad.device)
        scale = g_loss.detach().reshape(1)
        if scale.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            scale = scale.float()
        L.check(L.lib().aa_tail_scatter_scaled(grad.data_ptr(), L.dtype_code(grad.dtype), grad.stride(0), lens_dev.data_ptr(), B, W,
                                               ctx.src_width, scale.data_ptr(), L.dtype_code(scale.dtype), out.data_ptr(),
                                               out.stride(0), Lq, L.stream_ptr(grad.device)))
        return out.view(ctx.shape), None, None, None, None, None, None, None


def _loss_inputs(x, old, aux, mask):
    L.require_cuda(x, old, aux, mask)
    if not (x.shape == old.shape == aux.shape == mask.shape) or x.dim() != 2:
        raise ValueError('loss inputs must all be (B, W)')
    x = _contiguous_last(x)
    old = _contiguous_last(old.detach().to(x.dtype))
    aux = _contiguous_last(aux.detach())
    if aux.dtype not in (torch.float32, torch.bfloat16, torch.float16):
        aux = aux.float()
    mask = _contiguous_last(mask.to(torch.bool))
    return x, old, aux, mask


def actor_loss(log_probs, old_log_probs, advantages, mask, clip_range_ratio: float, mode: str | None = None):
    """PPOTrainer.actor_loss_fn (trainers/text_to_text/ppo.py:291-307), differentiable in log_probs."""
    x, old, aux, m = _loss_inputs(log_probs, old_log_probs, advantages, mask)
    loss, _, _ = _PpoLossFn.apply(x, old, aux, m, clip_range_ratio, _mode_code(mode, x.dtype), True)
    return loss


def critic_loss(values, old_values, returns, mask, clip_range_value: float, mode: str | None = None,
                return_row_mean: bool = False):
    """PPOTrainer.critic_loss_fn (trainers/text_to_text/ppo.py:510-526), differentiable in values."""
    x, old, aux, m = _loss_inputs(values, old_values, returns, mask)
    loss, row_mean, _ = _PpoLossFn.apply(x, old, aux, m, clip_range_value, _mode_code(mode, x.dtype), False)
    return (loss, row_mean) if return_row_mean else loss


def tail_actor_loss(logits: torch.Tensor, input_ids: torch.Tensor, lens, old_log_probs, advantages, mask,
                    clip_range_ratio: float, mode: str | None = None):
    """response_tail_log_probs + actor_loss as one autograd node (see _TailActorLossFn).
    -> (actor loss, new log-probs (B, W), the loss as fp32[2] for ppo_pack_metrics)."""
    L.require_cuda(logits, input_ids, old_log_probs, advantages, mask)
    lens = as_device_lens(lens, logits.device)
    B, K, _ = logits.shape
    if lens.bound > K - 1:
        raise ValueError(f'the logits tile holds {K} positions: too few for responses of up to {lens.bound} tokens')
    if not (tuple(old_log_probs.shape) == tuple(advantages.shape) == tuple(mask.shape) == (B, lens.bound)):
        raise ValueError('old_log_probs, advantages and mask must all be (B, W), W = the bound of the response lengths')
    logits, ids = _contiguous_last(logits), input_ids.contiguous()
    mode_code = _mode_code(mode, logits.dtype)
    lp_dtype = logits.dtype if mode_code == L.MODE_FAITHFUL else torch.float32
    old = _contiguous_last(old_log_probs.detach().to(lp_dtype))
    aux = _contiguous_last(advantages.detach())
    if aux.dtype not in (torch.float32, torch.bfloat16, torch.float16):
        aux = aux.float()
    m = _contiguous_last(mask.to(torch.bool))
    plan = device_tail_plan(lens, K, logits.stride(0), logits.stride(1), ids.stride(0), ids.size(1), 0, -1, lens.bound)
    return _TailActorLossFn.apply(logits, ids, plan, old, aux, m, clip_range_ratio, mode_code)


@functools.lru_cache(maxsize=64)
def _dense_actor_plan(B: int, L: int, start: int, sb: int, sl: int, lab_sb: int, device_str: str) -> RowPlan:
    """One segment per sample: rows [start, L - 1) of the (B, L, V) tile against labels ids[b, start + 1 :]."""
    W = L - 1 - start
    return RowPlan([b * sb + start * sl for b in range(B)], [b * lab_sb + start + 1 for b in range(B)],
                   [b * W for b in range(B)], [W] * B, [b * L + start for b in range(B)], (B, W), B * L,
                   torch.device(device_str))


def dense_actor_loss(logits: torch.Tensor, input_ids: torch.Tensor, start: int, old_log_probs, advantages, mask,
                     clip_range_ratio: float, mode: str | None = None):
    """The actor half of the text rl_step (trainers/text_to_text/ppo.py:336-349) as one autograd node:
    `gather_log_probabilities(logits[:, :-1], ids[:, 1:])[:, start:]` -> `actor_loss_fn` -> backward up to d logits.
    Only the rows `[start, L - 1)` are read (the reference scores every position and slices afterwards); with a
    gradient and rows long enough (see _single_pass_ok) the node is the single-pass K1f (see _TailActorLossFn), otherwise the
    composed ops gather_log_probabilities -> actor_loss.  old_log_probs / advantages / mask: (B, L - 1 - start).
    -> (actor loss, new log-probs (B, L - 1 - start), the loss for ppo_pack_metrics: fp32[2] buffer or the 0-dim loss)."""
    L.require_cuda(logits, input_ids, old_log_probs, advantages, mask)
    if logits.dim() != 3 or input_ids.shape != logits.shape[:2]:
        raise ValueError('expected logits (B, L, V) and input_ids (B, L)')
    B, Lq, _ = logits.shape
    start = int(start)
    W = Lq - 1 - start
    if start < 0 or W <= 0:
        raise ValueError(f'start = {start} leaves no scored position in a sequence of {Lq}')
    if not (tuple(old_log_probs.shape) == tuple(advantages.shape) == tuple(mask.shape) == (B, W)):
        raise ValueError('old_log_probs, advantages and mask must all be (B, L - 1 - start)')
    if not (_FUSED_ACTOR and _single_pass_ok(logits) and torch.is_grad_enabled() and logits.requires_grad):
        # short rows, fp16, no gradient: the composed ops (K1 over the response rows -> K5; backward K1b)
        lp = gather_log_probabilities(logits[:, start:-1], input_ids[:, start + 1:], mode=mode)
        loss = actor_loss(lp, old_log_probs, advantages, mask, clip_range_ratio, mode=mode)
        return loss, lp.detach(), loss
    logits, ids = _contiguous_last(logits), input_ids.contiguous()
    if B > 1 and (logits.stride(0) != Lq * logits.stride(1)):
        logits = logits.contiguous()  # the gradient tile is shaped after the logits: rows must be uniformly strided
    mode_code = _mode_code(mode, logits.dtype)
    lp_dtype = logits.dtype if mode_code == L.MODE_FAITHFUL else torch.float32
    old = _contiguous_last(old_log_probs.detach().to(lp_dtype))
    aux = _contiguous_last(advantages.detach())
    if aux.dtype not in (torch.float32, torch.bfloat16, torch.float16):
        aux = aux.float()
    m = _contiguous_last(mask.to(torch.bool))
    plan = _dense_actor_plan(B, Lq, start, logits.stride(0), logits.stride(1), ids.stride(0), str(logits.device))
    return _TailActorLossFn.apply(logits, ids, plan, old, aux, m, clip_range_ratio, mode_code)


def tail_critic_loss(scores: torch.Tensor, lens, old_values, returns, mask, clip_range_value: float,
                     mode: str | None = None):
    """critic_loss on `pad_sequence([scores.squeeze(-1)[b, :-1][-R_b:]])` without materialising that tensor (see
    _TailCriticLossFn).  scores (B, L, 1) or (B, L).  -> (critic loss, masked row means of the new values, loss fp32[2])."""
    L.require_cuda(scores, old_values, returns, mask)
    lens = as_device_lens(lens, scores.device)
    B = scores.size(0)
    if not (tuple(old_values.shape) == tuple(returns.shape) == tuple(mask.shape) == (B, lens.bound)):
        raise ValueError('old_values, returns and mask must all be (B, W), W = the bound of the response lengths')
    if lens.bound > scores.size(1) - 1:
        raise ValueError('the scores tensor is too short for the response lengths')
    x = scores if scores.dtype in (torch.float32, torch.bfloat16, torch.float16) else scores.float()
    old = _contiguous_last(old_values.detach().to(x.dtype))
    aux = _contiguous_last(returns.detach())
    if aux.dtype not in (torch.float32, torch.bfloat16, torch.float16):
        aux = aux.float()
    m = _contiguous_last(mask.to(torch.bool))
    return _TailCriticLossFn.apply(x, lens.dev, lens.bound, old, aux, m, clip_range_value, _mode_code(mode, x.dtype))


def ppo_pack_metrics(row_stats, reward, value_row_mean, actor_loss_t, critic_loss_t, coll=None) -> torch.Tensor:
    """The ten local metric scalars of trainers/text_to_text/ppo.py:360-381 as ONE fp32[12] vector
    (entries 0..8 AVG-reduced, entry 9 MAX-reduced).  With `coll` (FusedPackedAllReduce.next((9,))) the same
    kernel also performs that reduction over NVLink peer memory."""
    import ctypes

    dev = row_stats.device
    B = row_stats.size(0)
    stats = torch.empty(12, dtype=torch.float32, device=dev)
    a, c = actor_loss_t.detach(), critic_loss_t.detach()  # 0-dim losses or the fp32[2] buffers of the fused loss nodes
    a = a if (a.dtype == torch.float32 and a.dim() == 1) else a.float().reshape(1).contiguous()
    c = c if (c.dtype == torch.float32 and c.dim() == 1) else c.float().reshape(1).contiguous()
    L.check(L.lib().aa_ppo_pack_metrics(row_stats.data_ptr(), reward.detach().float().contiguous().data_ptr(),
                                        L.ptr(value_row_mean), a.data_ptr(), c.data_ptr(), B, stats.data_ptr(),
                                        ctypes.byref(coll) if coll is not None else None,
                                        _device_scratch(dev)['status'].data_ptr(), L.stream_ptr(dev)))
    return stats


# ---- integer layout ------------------------------------------------------------------------------
def move_padding_left(input_tensor: torch.Tensor, padding_value: int = 0) -> torch.Tensor:
    """trainers/text_image_to_text/ppo.py:56-87 / utils/tools.py:615-639, bit-exact, one launch."""
    L.require_cuda(input_tensor)
    if input_tensor.dim() != 2 or input_tensor.dtype != torch.int64:
        raise ValueError('move_padding_left expects an int64 (B, L) tensor')
    x = _contiguous_last(input_tensor)
    out = torch.empty(x.shape, dtype=torch.int64, device=x.device)
    L.check(L.lib().aa_move_padding_left(x.data_ptr(), x.size(0), x.size(1), x.stride(0), int(padding_value),
                                         out.data_ptr(), L.stream_ptr(x.device)))
    return out


class _TailRowsFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, lens_dev, rmax):
        B, W = x.shape
        out = torch.empty((B, rmax), dtype=x.dtype, device=x.device)
        L.check(L.lib().aa_tail_rows(x.data_ptr(), L.dtype_code(x.dtype), x.stride(0), lens_dev.data_ptr(), B, W, rmax,
                                     out.data_ptr(), out.stride(0), 0, L.stream_ptr(x.device)))
        ctx.save_for_backward(lens_dev)
        ctx.W = W
        return out

    @staticmethod
    def backward(ctx, g):
        (lens_dev,) = ctx.saved_tensors
        g = _contiguous_last(g)
        B, rmax = g.shape
        out = torch.empty((B, ctx.W), dtype=g.dtype, device=g.device)
        L.check(L.lib().aa_tail_rows(g.data_ptr(), L.dtype_code(g.dtype), g.stride(0), lens_dev.data_ptr(), B, ctx.W, rmax,
                                     out.data_ptr(), out.stride(0), 1, L.stream_ptr(g.device)))
        return out, None, None


def tail_rows(x: torch.Tensor, lens: Sequence[int]) -> torch.Tensor:
    """pad_sequence([x[b][-R_b:] for b], batch_first=True) for a (B, W) tensor
    (trainers/text_image_to_text/ppo.py:233-249, 318-330) in one launch, differentiable in x."""
    L.require_cuda(x)
    if isinstance(lens, DeviceLens):  # lengths on the device: the width is the host-known bound
        if x.dim() != 2 or len(lens) != x.size(0) or not 0 < lens.bound <= x.size(1):
            raise ValueError('tail_rows: x must be (B, W) with 0 <= R_b <= bound <= W')
        return _TailRowsFn.apply(_contiguous_last(x), lens.dev, lens.bound)
    lens = tuple(int(r) for r in lens)
    if x.dim() != 2 or len(lens) != x.size(0) or not 0 < max(lens) <= x.size(1) or min(lens) < 0:
        raise ValueError('tail_rows: x must be (B, W) with 0 <= R_b <= W')
    return _TailRowsFn.apply(_contiguous_last(x), _lens_tensor(lens, str(x.device)), max(lens))


def rollout_layout(prompt_ids: torch.Tensor, sequences: torch.Tensor, pad_id: int):
    """Everything trainers/text_image_to_text/ppo.py:185-203 does after `generate`, ONE launch, no host sync:
    -> (move_padding_left(sequences), its attention mask, DeviceLens of the response lengths).  The bound of the
    lengths is the number of generated positions (a response cannot be longer)."""
    L.require_cuda(prompt_ids, sequences)
    if prompt_ids.dim() != 2 or sequences.dim() != 2 or prompt_ids.size(0) != sequences.size(0) or \
            prompt_ids.dtype != torch.int64 or sequences.dtype != torch.int64:
        raise ValueError('rollout_layout expects int64 prompt_ids (B, P) and sequences (B, L)')
    p, x = _contiguous_last(prompt_ids), _contiguous_last(sequences)
    B, Lq = x.shape
    moved = torch.empty((B, Lq), dtype=torch.int64, device=x.device)
    mask = torch.empty((B, Lq), dtype=torch.bool, device=x.device)
    lens = torch.empty(B, dtype=torch.int32, device=x.device)
    L.check(L.lib().aa_ppo_rollout_layout(p.data_ptr(), p.size(1), p.stride(0), x.data_ptr(), Lq, x.stride(0), B, int(pad_id),
                                          moved.data_ptr(), mask.data_ptr(), lens.data_ptr(), L.stream_ptr(x.device)))
    return moved, mask, DeviceLens(lens, max(Lq - p.size(1), 1))


def response_tail_log_probs(logits: torch.Tensor, input_ids: torch.Tensor, lens, mode: str | None = None) -> torch.Tensor:
    """The multimodal PPO scoring rows (trainers/text_image_to_text/ppo.py:229-246, 296-309): sample b scores
    `logits[b, :-1][-R_b:]` against `input_ids[b, 1:][-R_b:]`, right-padded with 0 to (B, W), W = the lengths' bound.
    `logits` is (B, K, V) with K <= L: the LAST K positions of the sequences (K = L: the whole tile; K = W + 1: the
    `logits_to_keep` tail tile).  The labels are read in place from input_ids, the row plan is built on the device."""
    L.require_cuda(logits, input_ids)
    lens = as_device_lens(lens, logits.device)
    B, K, _ = logits.shape
    if input_ids.shape[0] != B or len(lens) != B or K > input_ids.size(1):
        raise ValueError('response_tail_log_probs: logits (B, K, V), input_ids (B, L >= K), one length per sample')
    if lens.bound > K - 1:
        raise ValueError(f'the logits tile holds {K} positions: too few for responses of up to {lens.bound} tokens')
    logits, ids = _contiguous_last(logits), input_ids.contiguous()
    plan = device_tail_plan(lens, K, logits.stride(0), logits.stride(1), ids.stride(0), ids.size(1), 0, -1, lens.bound)
    return _LogProbFn.apply(logits, ids, plan, _mode_code(mode, logits.dtype))


_DUAL_K1 = os.environ.get('AA_B200_DUAL_K1', '1') != '0'  # actor + reference rollout scoring in ONE K1 launch (bit-identical, ~1% of the PPO step)


def response_tail_log_probs_pair(logits_a: torch.Tensor, logits_b: torch.Tensor, input_ids: torch.Tensor, lens,
                                 mode: str | None = None):
    """response_tail_log_probs of TWO logits tensors of identical shape / dtype / strides against the same labels (the
    rollout's actor and reference model, text_image_to_text/ppo.py:229-246) in ONE K1 launch: the second tensor is
    addressed relative to the first one's base pointer.  No gradient.  -> (log_probs_a, log_probs_b), each (B, W)."""
    L.require_cuda(logits_a, logits_b, input_ids)
    lens = as_device_lens(lens, logits_a.device)
    a, b = _contiguous_last(logits_a.detach()), _contiguous_last(logits_b.detach())
    if a.shape != b.shape or a.dtype != b.dtype or a.stride() != b.stride():
        raise ValueError('both logits tensors must share shape, dtype and strides')
    B, K, _ = a.shape
    if lens.bound > K - 1:
        raise ValueError(f'the logits tile holds {K} positions: too few for responses of up to {lens.bound} tokens')
    delta = b.data_ptr() - a.data_ptr()
    if delta % a.element_size():
        raise ValueError('logits tensors are not element-aligned relative to each other')
    ids = input_ids.contiguous()
    plan = device_tail_plan(lens, K, a.stride(0), a.stride(1), ids.stride(0), ids.size(1), 0, -1, lens.bound, 2,
                            delta // a.element_size())
    mode_code = _mode_code(mode, a.dtype)
    out = torch.zeros(plan.out_shape, dtype=a.dtype if mode_code == L.MODE_FAITHFUL else torch.float32, device=a.device)
    _launch_fwd(a, ids, plan, out, None, None)
    return out[0], out[1]


def count_nonpad(ids: torch.Tensor, pad_id: int) -> torch.Tensor:
    """Per-row number of tokens != pad (int32, on device): the bookkeeping behind
    trainers/text_image_to_text/ppo.py:190-203 without the per-sample `.tolist()`."""
    L.require_cuda(ids)
    x = _contiguous_last(ids)
    out = torch.empty(x.size(0), dtype=torch.int32, device=x.device)
    L.check(L.lib().aa_count_nonpad(x.data_ptr(), x.size(0), x.size(1), x.stride(0), int(pad_id), out.data_ptr(),
                                    L.stream_ptr(x.device)))
    return out
