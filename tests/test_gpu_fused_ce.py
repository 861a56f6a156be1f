"""The causal-LM cross-entropy from the last hidden states (ops.causal_lm_loss_from_hidden[_scaled], ops.ce_rows) and the
trainers that use it with `fused_lm_head` (SupervisedTrainer.loss, PPOTrainer.ptx_step), on the B200: against the logits
path (ops.causal_lm_loss on F.linear), the oracle port on ATen CUDA and a real HF causal LM."""
from types import SimpleNamespace

import pytest
import torch
import torch.nn.functional as F

from oracle import ref_port as O

pytestmark = pytest.mark.gpu

DEV = 'cuda'


@pytest.fixture(scope='module')
def ops():
    if not torch.cuda.is_available():
        pytest.skip('needs a CUDA device')
    from align_anything_b200 import ops as _ops

    return _ops


def _labels(B, L, V, pattern, gen):
    labels = torch.randint(0, V, (B, L), generator=gen)
    if pattern == 'masked':  # prompt prefix, right pads, an interior ignored token
        for b in range(B):
            labels[b, : 5 + 7 * b] = -100
            labels[b, L - 3 * b:] = -100
        labels[0, L // 2] = -100
    elif pattern == 'single':  # exactly one valid shifted label
        labels[:] = -100
        labels[B - 1, L // 3] = int(torch.randint(0, V, (1,), generator=gen))
    elif pattern == 'none':
        labels[:] = -100
    return labels.to(DEV)


def _grad_close(got, want, what, k_len):
    """d(hidden) / d(weight) of the fused path against the logits path's.  Both are fp32-accumulated GEMMs over the same
    math, rounded to the operand dtype: half an ulp each, the truncating accumulation drift of the tensor cores over
    k_len / 16 additions (test_lm_head_backward_gemms_vs_matmul), and the d(logits) entries that come out one bf16 ulp
    apart because the two paths round logits computed in different summation orders (a few percent of the entries,
    random signs: a few 1e-3 of the largest value of a long reduction).  The scale is the largest |value|, not the rms:
    with one valid row d(hidden) is zero everywhere else."""
    assert got.shape == want.shape and got.dtype == want.dtype, what
    g, w = got.float(), want.float()
    assert not bool(torch.isnan(g).any()), what
    scale = float(w.abs().max())
    ulp = 2 ** -8 if got.dtype == torch.bfloat16 else 2 ** -22
    tol = 2 * ulp * w.abs() + (max(1e-4, (k_len / 16) * 2 ** -23) + (4e-3 if got.dtype == torch.bfloat16 else 1e-5)) * scale
    err = (g - w).abs()
    assert bool((err <= tol).all()), (what, float((err - tol).max()), int((err > tol).sum()), scale)


SHAPES = [  # (H, V, dtype, chunk_rows): K6 / K6b path, odd vocabularies, several d(logits) chunks, library fallbacks
    (64, 1031, torch.bfloat16, None),
    (128, 32064, torch.bfloat16, 128),
    (4096, 128257, torch.bfloat16, None),
    (48, 1031, torch.bfloat16, None),   # H % 64 != 0: chunked library GEMMs + K1 / K1b
    (64, 1031, torch.float32, 64),      # fp32 operands: the same fallback, several chunks
]


@pytest.mark.parametrize('pattern', ['masked', 'single', 'none'])
@pytest.mark.parametrize('shape', SHAPES, ids=lambda s: f'H{s[0]}-V{s[1]}-{str(s[2])[6:]}-c{s[3]}')
def test_loss_from_hidden_matches_the_logits_path(ops, shape, pattern):
    H, V, dtype, chunk = shape
    B, L = 3, 120
    gen = torch.Generator().manual_seed(H + V + len(pattern))
    h0 = torch.randn(B, L, H, generator=gen).to(dtype).to(DEV)
    w0 = (torch.randn(V, H, generator=gen) * (2.0 / H ** 0.5)).to(dtype).to(DEV)
    labels = _labels(B, L, V, pattern, gen)
    scale, g_in = 3.0, 0.5

    h, w = h0.clone().requires_grad_(True), w0.clone().requires_grad_(True)
    scaled, loss = ops.causal_lm_loss_from_hidden_scaled(h, w, labels, scale, chunk_rows=chunk)
    assert scaled.dtype == loss.dtype == torch.float32 and not loss.requires_grad
    scaled.backward(torch.tensor(g_in, device=DEV))
    hr, wr = h0.clone().requires_grad_(True), w0.clone().requires_grad_(True)
    want_scaled, want = ops.causal_lm_loss_scaled(F.linear(hr, wr), labels, scale)
    want_scaled.backward(torch.tensor(g_in, device=DEV))
    plain = ops.causal_lm_loss_from_hidden(h0, w0, labels, chunk_rows=chunk)
    ops.check_status(DEV)
    if pattern == 'none':
        assert torch.isnan(loss) and torch.isnan(want) and torch.isnan(plain)
        assert torch.count_nonzero(h.grad) == 0 and torch.count_nonzero(w.grad) == 0
        return
    # the bar is set on logits accumulated in fp32 and rounded once (what the lm_head's tensor-core GEMM computes); the
    # library GEMM behind F.linear is held to it too except at an odd vocabulary, where cuBLAS runs its unaligned
    # kernels and their bf16 logits drift by more (DESIGN.md section 8)
    exact = F.linear(h0.float(), w0.float()).to(dtype)
    checks = [(ops.causal_lm_loss(exact, labels), 2e-5, 'logits path, exact logits'),
              (O.causal_lm_loss(exact, labels), 2e-5, 'oracle port, exact logits'),
              (want, 2e-5 if V % 2 == 0 else 1e-4, 'logits path, F.linear'),
              (O.causal_lm_loss(F.linear(h0, w0), labels), 2e-5 if V % 2 == 0 else 1e-4, 'oracle port, F.linear')]
    for ref, rtol, what in checks:
        assert abs(float(loss) - float(ref)) <= rtol * abs(float(ref)), (what, float(loss), float(ref))
    assert abs(float(scaled.detach()) - scale * float(loss)) <= 1e-6 * abs(float(scaled.detach()))
    assert float(plain) == float(loss)
    # gradients: against the logits path on the same exactly-accumulated logits, its d(logits) taken through fp32 GEMMs
    # (at V = 128257 the library's own d(hidden) GEMM runs on an odd leading dimension and drifts by more); at an even
    # vocabulary also against the plain F.linear path
    he, we = h0.float().requires_grad_(True), w0.float().requires_grad_(True)
    ops.causal_lm_loss_scaled(F.linear(he, we).to(dtype), labels, scale)[0].backward(torch.tensor(g_in, device=DEV))
    refs = [(he.grad.to(dtype), we.grad.to(dtype), 'exact logits')] + ([(hr.grad, wr.grad, 'F.linear')] if V % 2 == 0 else [])
    for dh_want, dw_want, what in refs:
        _grad_close(h.grad, dh_want, f'd hidden {shape} {pattern} vs {what}', V)
        _grad_close(w.grad, dw_want, f'd weight {shape} {pattern} vs {what}', B * L)
    # rows whose shifted label is ignored get exactly-zero d(hidden)
    shift = torch.full_like(labels, -100)
    shift[:, :-1] = labels[:, 1:]
    assert float(h.grad[shift == -100].abs().max()) == 0.0


def _ce_rows_reference(labels, ignore_index):
    shift = torch.full_like(labels, ignore_index)
    shift[:, :-1] = labels[:, 1:]
    flat = shift.reshape(-1)
    idx = torch.nonzero(flat != ignore_index).reshape(-1)
    return idx, flat[idx]


@pytest.mark.parametrize('B,L,p_valid', [(1, 7, 0.5), (4, 1000, 0.3), (7, 2051, 0.9), (3, 4096, 0.02)])
def test_ce_rows_compaction(ops, B, L, p_valid):
    gen = torch.Generator().manual_seed(B * L)
    V = 32064
    base = torch.randint(0, V, (B, 2 * L), generator=gen)
    base[torch.rand(B, 2 * L, generator=gen) >= p_valid] = -100
    labels = base.to(DEV)[:, ::2]  # strided: the kernel takes both label strides
    for lab in (labels, labels.contiguous()):
        rows = ops.ce_rows(lab, V)
        idx, want = _ce_rows_reference(lab, -100)
        assert rows.n_valid() == idx.numel()
        assert torch.equal(rows.index, idx) and torch.equal(rows.labels, want)
    ops.check_status(DEV)


def test_ce_rows_out_of_range_label_sets_the_status_word(ops):
    from align_anything_b200 import _lib as L

    labels = torch.full((2, 16), -100, dtype=torch.int64, device=DEV)
    labels[0, 3], labels[1, 9] = 5, 1031  # 1031 == V: outside [0, V)
    rows = ops.ce_rows(labels, 1031)
    assert rows.n_valid() == 2
    with pytest.raises(IndexError, match='outside'):
        ops.check_status(DEV)
    labels[1, 9] = -7
    ops.ce_rows(labels, 1031).n_valid()
    status = int(ops.status_lane(DEV).item())
    assert status & L.STATUS_LABEL_OOB
    with pytest.raises(IndexError):
        ops.raise_for_status(status, DEV)
    ops.check_status(DEV)  # the word was reset


class _Engine:
    def __init__(self, model):
        self.module = model
        self.optimizer = SimpleNamespace(param_groups=[{'lr': 1e-5}])

    def __call__(self, **kw):
        return self.module(**kw)

    def backward(self, loss):
        loss.backward()

    def step(self):
        pass

    def get_output_embeddings(self):
        return self.module.get_output_embeddings()


def _tiny_llama(tie):
    from transformers import LlamaConfig, LlamaForCausalLM

    torch.manual_seed(5)
    cfg = LlamaConfig(vocab_size=1031, hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=4,
                      num_key_value_heads=2, tie_word_embeddings=tie, max_position_embeddings=256)
    return LlamaForCausalLM(cfg).to(DEV, torch.bfloat16)


def _sft_batch(V=1031, B=3, L=48):
    gen = torch.Generator().manual_seed(9)
    ids = torch.randint(0, V, (B, L), generator=gen)
    mask = torch.ones(B, L, dtype=torch.bool)
    labels = ids.clone()
    for b, (prompt, pads) in enumerate(((9, 0), (14, 6), (5, 11))):
        labels[b, :prompt] = -100  # the prompt is not trained on
        if pads:
            ids[b, L - pads:], mask[b, L - pads:], labels[b, L - pads:] = 0, False, -100
    return {'input_ids': ids.to(DEV), 'attention_mask': mask.to(DEV), 'labels': labels.to(DEV)}


@pytest.mark.parametrize('tie', [False, True])
def test_sft_trainer_on_a_real_causal_lm(ops, tie):
    from align_anything_b200.trainers.text_to_text.sft import SupervisedTrainer

    model = _tiny_llama(tie)
    batch = _sft_batch()
    with torch.no_grad():
        own = model(**batch).loss  # transformers' ForCausalLMLoss on the model's own logits
    grads, losses = {}, {}
    for fused in (False, True):
        model.zero_grad(set_to_none=True)
        tr = SupervisedTrainer(None, _Engine(model))
        tr.fused_lm_head = fused
        loss = tr.loss(batch)['loss']
        loss.backward()
        losses[fused] = float(loss.detach())
        grads[fused] = {n: p.grad.detach().clone() for n, p in model.named_parameters()}
    ops.check_status(DEV)
    for fused in (False, True):
        assert abs(losses[fused] - float(own)) <= 2e-5 * abs(float(own)), (fused, losses[fused], float(own))
    assert abs(losses[True] - losses[False]) <= 2e-5 * abs(losses[False])
    if tie:
        assert model.lm_head.weight is model.model.embed_tokens.weight
    for name, want in grads[False].items():
        got = grads[True][name]
        rel = float((got.float() - want.float()).norm() / want.float().norm().clamp_min(1e-30))
        assert rel <= 2e-2, (name, rel)
    # the tied matrix collects both uses: embedding rows of the batch's tokens AND the lm_head gradient
    head = 'model.embed_tokens.weight' if tie else 'lm_head.weight'
    assert torch.count_nonzero(grads[True][head]) > 0


class _HiddenStatesModel:
    """A causal LM stand-in whose last hidden states are a leaf: logits when asked for them, hidden states with
    `output_hidden_states=True`; `strict` asserts that the fused path never asks for logits."""

    def __init__(self, h, w, strict, takes_keep=True):
        self.h, self.w, self.strict, self.takes_keep = h, w, strict, takes_keep
        self.calls = []

    def __call__(self, input_ids=None, attention_mask=None, **kw):
        self.calls.append(dict(kw))
        if 'labels' in kw:
            raise AssertionError('the loss is not computed inside the model')
        if 'logits_to_keep' in kw and not self.takes_keep:
            raise TypeError("forward() got an unexpected keyword argument 'logits_to_keep'")
        if self.strict:
            assert kw == {'output_hidden_states': True, 'logits_to_keep': 1}, kw
        hidden = self.h * 1.0
        if kw.get('output_hidden_states'):
            return SimpleNamespace(hidden_states=(hidden,), logits=F.linear(hidden[:, -1:], self.w))
        return SimpleNamespace(logits=F.linear(hidden, self.w))

    def get_output_embeddings(self):
        return SimpleNamespace(weight=self.w)


def _leaves(H=128, V=32064, B=2, L=64, seed=3):
    gen = torch.Generator().manual_seed(seed)
    h = torch.randn(B, L, H, generator=gen).bfloat16().to(DEV)
    w = (torch.randn(V, H, generator=gen) * 0.15).bfloat16().to(DEV)
    labels = _labels(B, L, V, 'masked', gen)
    return h, w, labels


def test_multimodal_ptx_step_with_fused_lm_head(ops):
    from align_anything_b200.trainers.text_image_to_text.ppo import PPOTrainer

    h0, w0, labels = _leaves()
    batch = {'input_ids': labels.clamp(min=0), 'attention_mask': labels != -100, 'labels': labels}
    res = {}
    for fused in (False, True):
        h, w = h0.clone().requires_grad_(True), w0.clone().requires_grad_(True)
        model = _HiddenStatesModel(h, w, strict=fused)
        t = object.__new__(PPOTrainer)
        t.infer_batch = lambda b: {k: v for k, v in b.items() if k != 'meta_info'}
        t.actor_model, t.ptx_coeff, t.fused_lm_head = _Engine(model), 16.0, fused
        out = t.ptx_step(batch)
        assert model.calls and all(('logits_to_keep' in c) == fused for c in model.calls)
        res[fused] = (out['train/ptx_loss'], h.grad, w.grad)
    ops.check_status(DEV)
    (l0, hg0, wg0), (l1, hg1, wg1) = res[False], res[True]
    assert abs(l1 - l0) <= 2e-5 * abs(l0), (l1, l0)
    _grad_close(hg1, hg0, 'ptx d hidden', w0.size(0))
    _grad_close(wg1, wg0, 'ptx d weight', h0.size(0) * h0.size(1))


def test_forward_without_logits_to_keep_gives_the_logits_path_loss(ops):
    from align_anything_b200.trainers.text_to_text.sft import SupervisedTrainer

    h0, w0, labels = _leaves(seed=4)
    batch = {'input_ids': labels.clamp(min=0), 'attention_mask': labels != -100, 'labels': labels}
    want = float(ops.causal_lm_loss(F.linear(h0, w0), labels))
    tr = SupervisedTrainer(None, _Engine(_HiddenStatesModel(h0, w0, strict=False, takes_keep=False)))
    tr.fused_lm_head = True
    with pytest.warns(RuntimeWarning, match='logits_to_keep'):
        got = float(tr.loss(batch)['loss'])
    assert tr.fused_lm_head is False
    assert abs(got - want) <= 1e-6 * abs(want), (got, want)
    ops.check_status(DEV)
